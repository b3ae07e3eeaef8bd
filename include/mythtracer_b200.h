/* mythtracer_b200 -- C ABI of the B200-native (sm_100a) replacement for MythTracer's ray-casting hot path.
 *
 * The reference has no plugin/FFI layer: its boundary for this path is the public C++ API of
 * `raytracer::MythTracer` (reference VerStarting/mythtracer.h:55-66) together with the public members of
 * Scene / OctTree / Camera / Light / Material / WorkChunk.  This header is the thin `extern "C"` layer that
 * boundary is re-implemented on (plain pointers and sizes, no C++ or torch types); the header-compatible
 * C++ classes in include/mythtracer/ and the Python mirror in mythtracer_b200/api.py are written on top of
 * it, and INTEGRATION.md shows how a maintainer of the reference binds it.
 *
 * There is NO CPU fallback: every entry point that renders or intersects runs hand-written CUDA kernels
 * and fails with MTB_ERR_CUDA when no sm_100 device is usable.
 *
 * Struct layouts mirror the reference's data members one to one (same order, FP64 throughout).
 */
#ifndef MYTHTRACER_B200_H_
#define MYTHTRACER_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MTB_OK 0
#define MTB_ERR_ARG (-1)      /* bad argument / bad state (e.g. render before a scene is uploaded) */
#define MTB_ERR_CUDA (-2)     /* CUDA runtime error; text in mtb_last_error() */
#define MTB_ERR_IO (-3)       /* loader: file missing or malformed (the reference's `return false` paths) */
#define MTB_ERR_LIMIT (-4)    /* scene exceeds a documented limit (octree deeper than MTB_MAX_TREE_DEPTH) */

#define MTB_MAX_TREE_DEPTH 48 /* the reference has no cap (octtree.cc:52-55); deeper trees are refused */
#define MTB_MAX_RAY_DEPTH 16  /* max_depth argument = the reference's MAX_RECURSION_LEVEL (mythtracer.h:11) */

typedef struct mtb_context mtb_context;

/* reference camera.h:31-33; byte-identical to what Camera::Serialize writes (camera.cc:71-81) */
typedef struct {
  double origin[3];
  double pitch, yaw, roll; /* degrees, X / Y / Z axis */
  double aov;              /* horizontal angle of view, degrees */
} mtb_camera;

/* reference light.h:8-14 */
typedef struct {
  double position[3], ambient[3], diffuse[3], specular[3];
} mtb_light;

/* reference material.h:12-48 (`Texture *tex` becomes an index into the texture table, -1 = none) */
typedef struct {
  double ambient[3], diffuse[3], specular[3]; /* Ka Kd Ks */
  double specular_exp;                        /* Ns */
  double reflectance;                         /* Refl */
  double transparency;                        /* Tr */
  double transmission_filter[3];              /* Tf */
  double refraction_index;                    /* Ni */
  int32_t texture;
  int32_t pad_;
} mtb_material;

/* 8-bit RGBA texels, row-major, top row first: what texture.cc:81-104 holds after SDL's RGBA32 conversion.
 * The px/255.0 conversion (texture.cc:100-104) happens on the device in FP64. */
typedef struct {
  int32_t width, height;
  const uint8_t *rgba;
} mtb_texture;

/* reference primitive_triangle.h:26-29 + primitive.h:41-42.  Array order = OctTree::AddPrimitive order
 * (octtree.cc:8-14); it decides ties exactly as the reference's list order does. */
typedef struct {
  double vertex[9];
  double normal[9];
  double uvw[9];
  int32_t material; /* index into the material table, -1 = `mtl == nullptr` */
  int32_t line_no;  /* Primitive::debug_line_no */
} mtb_triangle;

/* reference mythtracer.h:13-16 (PerPixelDebugInfo; 32 bytes on x86-64) */
typedef struct {
  int32_t line_no; /* -1 on a miss */
  int32_t pad_;
  double point[3]; /* NaN on a miss */
} mtb_debug;

/* Optional per-pixel decision taps (device-computed; used by the parity tests, see oracle/mt_oracle.h).  The sizes
 * below are those of mtb_render_chunk; mtb_render_batch_debug takes n_views * (s*image_h) * (s*image_w) entries. */
typedef struct {
  uint64_t *sig_hits;   /* chunk_w*chunk_h, may be NULL */
  uint64_t *sig_shadow; /* chunk_w*chunk_h, may be NULL */
  uint32_t *n_rays;     /* chunk_w*chunk_h, may be NULL */
} mtb_taps;

/* Thin-lens sample of one sub-frame of mtb_render_batch_lens: the lens point (u, v) in world units, u along the image's
 * right and v along its down direction, and the distance of the focal plane from the camera origin along its normal. */
typedef struct {
  double u, v;
  double focus_distance;
} mtb_lens;

/* Work done by one render / intersect call.  Counters other than `rays..refract` are only filled by the
 * counting build of the kernels (MTB_FLAG_COUNT_WORK), which is slower and never timed. */
typedef struct {
  uint64_t rays;     /* OctTree::IntersectRay-equivalent queries = primary + shadow + reflect + refract */
  uint64_t primary, shadow, reflect, refract;
  uint64_t n_slab;    /* octree child / root box tests */
  uint64_t n_visit;   /* octree nodes entered */
  uint64_t n_triaabb; /* exact triangle AABB pre-tests (primitive_triangle.cc:85-108) */
  uint64_t n_mt;      /* Moller-Trumbore evaluations */
  uint64_t n_hit;     /* triangle tests that returned true */
  uint64_t n_shade;   /* shaded hits */
  uint64_t n_bvh;     /* list-BVH box tests (no reference counterpart: they replace n_triaabb work) */
  uint64_t n_literal; /* rays that took the literal (NaN-exact) traversal */
  uint64_t n_fast;     /* rays answered by the certified fast traversal (scene BVH) */
  uint64_t n_fallback; /* rays the fast traversal could not certify and handed to the exact octree recursion */
  uint64_t n_long128_rays, n_long128_visits; /* fast traversals of more than 128 scene-BVH node visits, and their visits */
  uint64_t n_long512_rays, n_long512_visits; /* ... of more than 512 node visits (the tail that bounds small partitions) */
  double kernel_ms;   /* device time of the kernels of this call (CUDA events) */
  double total_ms;    /* host wall time of the call, copies included */
} mtb_stats;

typedef struct {
  int64_t n_triangles, n_nodes, n_bvh_nodes;
  int32_t tree_depth, n_materials, n_textures, n_lights;
  int64_t root_list, biggest_list, interior_triangles;
  double aabb_min[3], aabb_max[3]; /* OctTree::GetAABB (octtree.cc:42-44) */
  int64_t device_bytes;
  int64_t n_scene_refs; /* leaf positions of the scene BVH: >= n_triangles (large triangles are referenced from several leaves) */
} mtb_scene_summary;

#define MTB_FLAG_COUNT_WORK 1u   /* fill the n_* work counters (counting kernels) */
#define MTB_FLAG_NO_LIST_BVH 2u  /* scan every node list linearly, like the reference (A/B measurements) */
/* Pipeline choice.  With none of the pipeline bits set the library decides at run time: on the first frames of a
 * given geometry (chunk size, partition, depth, light count) it times the per-pixel megakernel (second frame, once
 * its cost-aware tile order is warm) and the queue pipeline (fourth frame, once its buffers exist) and keeps the
 * faster from frame 5 on.  Both produce identical bytes, so the choice is invisible in the output (DESIGN.md
 * section 6). */
#define MTB_FLAG_MEGAKERNEL 16u  /* force the per-pixel megakernel */
#define MTB_FLAG_QUEUE 8192u     /* force the queue pipeline: the wavefront as ONE persistent kernel over a single device-side ray queue (all levels) */
#define MTB_FLAG_WAVEFRONT 4u    /* the same as MTB_FLAG_QUEUE: the queue pipeline is the wavefront's only form */
#define MTB_FLAG_EXACT_OCTREE 128u /* every regular ray walks the octree in the reference's recursion order (no certified fast traversal) */
/* Retired forms (all bit-identical, all measured slower on B200; DESIGN.md sections 5, 6 and 11 keep the numbers).
 * The bits are still accepted and ignored, so callers that set them keep working. */
#define MTB_FLAG_HYBRID 2048u     /* was: hybrid frames, the most expensive tiles through the level-by-level wavefront, the rest through the megakernel */
#define MTB_FLAG_RAY_SORT 8u      /* was: wavefront, counting-sort every queue by origin cell + direction octant */
#define MTB_FLAG_PACKING 256u     /* was: megakernel, block-level ray packing on 16x8 tiles */
#define MTB_FLAG_RESUME 1024u     /* was: megakernel, suspendable walks */
#define MTB_FLAG_WARP_SYNC 512u   /* was: megakernel, forced warp re-convergence in front of every traversal */
#define MTB_FLAG_PERSISTENT 64u   /* was: megakernel, persistent warps drawing pixels from a counter */
#define MTB_FLAG_PAIR_RAYS 16384u /* was: mtb_intersect_rays, rays 2i and 2i+1 walked in lock step by one thread */
#define MTB_FLAG_CHAIN_RAYS 32768u /* was: mtb_intersect_rays, rays 2i and 2i+1 walked back to back in one node loop */
/* Scene BVH built ON THE DEVICE (PLOC over the reference boxes, csrc/device_build.cu; SURVEY section 8 f1) instead of
 * on the host threads (binned SAH).  Measured on B200, C3: the device build takes ~20-50 ms against 165 ms on 24 host
 * cores (time to first frame 0.31 s vs 0.39 s), but its trees cost 12 % more box tests per ray (frame 10.2 vs 9.17 ms):
 * the right choice for a scene that is rendered a few times, the wrong one for an animation - hence opt-in.  The
 * rendered bytes are the same either way. */
#define MTB_FLAG_DEVICE_BVH 4096u
#define MTB_FLAG_NO_TILE_ORDER 32u /* megakernel: always launch tiles in scanline order (A/B of the cost-aware launch order) */

/* ---- life cycle -------------------------------------------------------------------------------- */

/* Creates a context on `n_devices` CUDA devices (device ordinals in `devices`; NULL = device 0 only).
 * One host thread drives one context (the reference's MythTracer is not re-entrant either). */
int mtb_create(mtb_context **out, const int *devices, int n_devices);
/* A context without any device: the loader, the octree builder and the inspection calls work (host-side
 * logic can be tested on a machine without a GPU); every render / intersect call fails with MTB_ERR_CUDA. */
int mtb_create_host(mtb_context **out);
void mtb_destroy(mtb_context *ctx);
/* Text of the last error on this context (or of the last failed mtb_create when ctx == NULL). */
const char *mtb_last_error(const mtb_context *ctx);
int mtb_device_count(const mtb_context *ctx);

/* ---- scene ------------------------------------------------------------------------------------- */

/* Replaces OctTree::AddPrimitive + Finalize (octtree.cc:8-24,46-135) and the AoS Scene: builds the
 * reference's octree (same boxes, same list membership and order), flattens it and uploads SoA buffers to
 * every device of the context.  Lights are untouched. */
int mtb_scene_upload(mtb_context *ctx, const mtb_triangle *tris, int64_t n_tris, const mtb_material *mtls,
                     int32_t n_mtls, const mtb_texture *texs, int32_t n_texs);
/* MythTracer::LoadObj (mythtracer.cc:247-256): OBJ + MTL (+ PPM map_Ka textures) -> mtb_scene_upload. */
int mtb_load_obj(mtb_context *ctx, const char *path);
/* scene.lights (scene.h:14) -- the reference's callers rewrite it every frame (main_local.cc:79-110). */
int mtb_set_lights(mtb_context *ctx, const mtb_light *lights, int32_t n);
int mtb_scene_info(const mtb_context *ctx, mtb_scene_summary *out);
/* Copies out the host-side triangle / material tables the loader produced (NULL = skip). */
int mtb_scene_read(const mtb_context *ctx, mtb_triangle *tris, mtb_material *mtls);
/* What the loader kept besides the tables: names (MaterialMap / TextureMap keys, material.h:50, texture.h:25)
 * and the decoded RGBA32 texels.  Pointers stay valid until the next scene load on this context. */
const char *mtb_scene_material_name(const mtb_context *ctx, int32_t index);
const char *mtb_scene_texture_name(const mtb_context *ctx, int32_t index);
int mtb_scene_texture(const mtb_context *ctx, int32_t index, mtb_texture *out);
/* MtlFileReader::ReadMtlFile (objreader.cc:472-549): materials (+ textures) only, no geometry. */
int mtb_load_mtl(mtb_context *ctx, const char *path);
/* Octree membership of every triangle (insertion order): the box of the node whose list holds it
 * (6 doubles: lo.xyz, hi.xyz) and that node's depth.  Either pointer may be NULL. */
int mtb_scene_triangle_nodes(const mtb_context *ctx, double *node_box, int32_t *node_depth);
/* The scene BVH of the certified fast traversal (DESIGN.md section 4), for inspection: node count, depth, the
 * nodes themselves (64 bytes each: float lbox[6], rbox[6]; int32 left, right, pad[2]; a child >= 0 is a node
 * index, < 0 a leaf with ~child = (first << 3) | count over leaf_order) and, per leaf position, the insertion
 * index of the triangle stored there (mtb_scene_summary::n_scene_refs entries).  Any pointer may be NULL.  n_nodes == 0: the scene
 * has no fast traversal (empty scene, MTB_FLAG_NO_LIST_BVH, or a tree deeper than the traversal stack). */
int mtb_scene_bvh(const mtb_context *ctx, int64_t *n_nodes, int32_t *depth, void *nodes, int32_t *leaf_order);
/* Stages of the last scene load, milliseconds (time to the first frame, SURVEY.md section 8 f1): out_ms[0] OBJ + MTL
 * parse, [1] octree (AttemptSplit), [2] flatten + list BVHs, [3] scene BVH on the host (or just its references when
 * it is built on the device), [4] scene BVH on the device incl. the leaf-record gather, [5] upload, [6] 1.0 when
 * the scene BVH was built on the device, [7] the host tree build itself (it runs on its own thread while [1] and [2]
 * proceed; [3] is only what was left to wait for, plus the leaf-record gather). */
int mtb_load_timing(const mtb_context *ctx, double out_ms[8]);
int mtb_set_flags(mtb_context *ctx, uint32_t flags);
/* Tile partitioning across processes -- the in-process form of the reference's master/worker contract
 * (main_net_master.cc:195-221: the frame is cut into tiles, every worker holds the whole scene and renders
 * the tiles it is handed).  The chunk is cut into strips of 8 rows; with (part_index, part_count) this
 * context renders only the strips s with s % (part_count * n_devices) == part_index * n_devices + g on its
 * device g and leaves all other pixels of the output untouched.  Default (0, 1): everything. */
int mtb_set_partition(mtb_context *ctx, int part_index, int part_count);

/* ---- the hot path ------------------------------------------------------------------------------ */

/* MythTracer::RayTrace(WorkChunk*) (mythtracer.cc:280-312): renders chunk [chunk_x, chunk_x+chunk_w) x
 * [chunk_y, chunk_y+chunk_h) of an image_w x image_h frame.  rgb_out: HOST buffer, chunk_w*chunk_h*3
 * bytes, row-major RGB24, stride chunk_w*3 (WorkChunk::output_bitmap).  dbg_out (HOST, nullable):
 * chunk_w*chunk_h PerPixelDebugInfo (WorkChunk::output_debug).  taps / stats nullable.  max_depth is the
 * reference's compile-time MAX_RECURSION_LEVEL.  With several devices the chunk is split into
 * interleaved tile rows, rendered concurrently and gathered over NVLink peer copies. */
int mtb_render_chunk(mtb_context *ctx, const mtb_camera *cam, int image_w, int image_h, int chunk_x, int chunk_y,
                     int chunk_w, int chunk_h, int max_depth, uint8_t *rgb_out, mtb_debug *dbg_out,
                     const mtb_taps *taps, mtb_stats *stats);

/* Frame sequencing (reference main_local.cc:51-149 renders, then writes, then renders ...): the same render as
 * mtb_render_chunk, enqueued without waiting -- the call returns as soon as the kernels and the device->host copy
 * of the frame are queued (no pipeline reads anything back while a frame is in flight).  rgb_out
 * must stay valid until mtb_wait returns and should come from mtb_host_alloc (pinned memory) for the copy to be
 * asynchronous.  With two such buffers a driver writes frame k to disk while frame k+1 renders
 * (apps/mythtracer_local_b200.cc). */
int mtb_render_chunk_async(mtb_context *ctx, const mtb_camera *cam, int image_w, int image_h, int chunk_x, int chunk_y,
                           int chunk_w, int chunk_h, int max_depth, uint8_t *rgb_out);
/* Waits for everything queued on the context's devices. */
int mtb_wait(mtb_context *ctx);
/* Pinned host memory for mtb_render_chunk_async (NULL when the allocation fails). */
void *mtb_host_alloc(size_t bytes);
void mtb_host_free(void *p);

/* Batches: N whole frames of one scene, one camera and one light set per view, in one launch per device (an orbit, a
 * camera path, a light sweep, many small views: a 480x270 frame is less than one wave of the B200, a batch of them
 * fills the machine).  Always the per-pixel megakernel: the pipeline bits (MTB_FLAG_WAVEFRONT, _QUEUE,
 * _MEGAKERNEL) are ignored; MTB_FLAG_COUNT_WORK and the traversal flags apply as for a single frame.  The bytes of view
 * v equal those of mtb_render_chunk with cams[v] and view v's lights.  A batch leaves the state of the single-frame
 * path alone (the context's lights, the automatic pipeline choice, the tile order).  With several devices, device g
 * renders a contiguous range of the views (counts differ by at most one) and copies them to their slice of rgb_out;
 * there is no gather.  The partition must be (0, 1).
 *
 * rgb_out: HOST, n_views * image_h * image_w * 3 bytes, view-major.  lights: n_views * n_lights entries
 * (view v uses lights[v*n_lights .. +n_lights)); NULL = every view uses the context's lights (mtb_set_lights)
 * and n_lights is ignored.  n_views: 1..65535.  stats (nullable): summed over views; kernel_ms = slowest device. */
int mtb_render_batch(mtb_context *ctx, const mtb_camera *cams, int32_t n_views, const mtb_light *lights,
                     int32_t n_lights, int image_w, int image_h, int max_depth, uint8_t *rgb_out, mtb_stats *stats);
/* Same, returns once queued (rgb_out pinned, from mtb_host_alloc; mtb_wait joins), like mtb_render_chunk_async.
 * cams and lights may be reused as soon as the call returns. */
int mtb_render_batch_async(mtb_context *ctx, const mtb_camera *cams, int32_t n_views, const mtb_light *lights,
                           int32_t n_lights, int image_w, int image_h, int max_depth, uint8_t *rgb_out);

/* Supersampled (anti-aliased) batches: as mtb_render_batch, with s = samples_per_axis samples per axis of every
 * output pixel.  With F the frame mtb_render_batch renders for the same view at (s*image_w) x (s*image_h), output
 * pixel (x, y) channel c of a view is
 *     (sum over i, j in 0..s-1 of F[s*y + j][s*x + i][c] + s*s/2) / (s*s)      (integer division)
 * the mean of the reference's own quantised samples at its own sensor positions (no jitter), rounded half up.  The
 * means are formed in the kernel: no high-resolution frame is stored and there is no second kernel.
 *
 * samples_per_axis: 1, 2, 4 or 8 (anything else: MTB_ERR_ARG); 1 is exactly mtb_render_batch.  s*image_w and
 * s*image_h: at most 65536.  rgb_out: HOST, n_views * image_h * image_w * 3 bytes (output pixels), view-major.
 * stats: those of the (s*image_w) x (s*image_h) batch (rays and, under MTB_FLAG_COUNT_WORK, every work counter). */
int mtb_render_batch_ss(mtb_context *ctx, const mtb_camera *cams, int32_t n_views, const mtb_light *lights,
                        int32_t n_lights, int image_w, int image_h, int samples_per_axis, int max_depth, uint8_t *rgb_out,
                        mtb_stats *stats);
/* Same, returns once queued (rgb_out pinned, from mtb_host_alloc; mtb_wait joins). */
int mtb_render_batch_ss_async(mtb_context *ctx, const mtb_camera *cams, int32_t n_views, const mtb_light *lights,
                              int32_t n_lights, int image_w, int image_h, int samples_per_axis, int max_depth,
                              uint8_t *rgb_out);

/* Batches with per-pixel planes: mtb_render_batch_ss (synchronous), which also returns for every view what
 * mtb_render_chunk returns for a frame besides its bytes: the PerPixelDebugInfo of the primary hit (line_no and point,
 * -1 / NaN on a miss; WorkChunk::output_debug) and the taps.  The planes live on each view's sample grid, of
 * (s*image_w) x (s*image_h) entries: entry (x, y) of view v is exactly what mtb_render_chunk writes for pixel (x, y)
 * of an (s*image_w) x (s*image_h) frame rendered with cams[v] and view v's lights.  For s = 1 that is the view itself;
 * for s > 1 they are the planes of the samples (no per-output-pixel aggregate is formed).
 *
 * dbg_out and each pointer of taps (and taps itself) may be NULL; each non-NULL one is a HOST array of
 * n_views * (s*image_h) * (s*image_w) entries, view-major and row-major.  With every plane NULL the call is
 * mtb_render_batch_ss.  rgb_out and stats are those of the same call without planes, byte for byte.  Arguments,
 * limits and the partition rule are those of mtb_render_batch_ss.  With several devices every device copies the
 * planes of its own views; there is no gather.  The single-frame path's debug and tap buffers are not used. */
int mtb_render_batch_debug(mtb_context *ctx, const mtb_camera *cams, int32_t n_views, const mtb_light *lights,
                           int32_t n_lights, int image_w, int image_h, int samples_per_axis, int max_depth,
                           uint8_t *rgb_out, mtb_debug *dbg_out, const mtb_taps *taps, mtb_stats *stats);

/* Accumulated batches (motion blur, soft shadows from area lights): every output view is the mean of k = subframes
 * sub-frames, each with its own camera and light set.  Sub-frame u = v*k + j (j < k) of output view v uses cams[u]
 * and lights[u*n_lights .. +n_lights).  With F_u the frame mtb_render_batch renders for sub-frame u at
 * (s*image_w) x (s*image_h), s = samples_per_axis, output pixel (x, y) channel c of view v is
 *     (sum over j < k, a, b < s of F_{v*k+j}[s*y + b][s*x + a][c] + k*s*s/2) / (k*s*s)      (integer division)
 * the rounded-half-up mean of all k*s*s quantised samples (not a mean of per-sub-frame means).  The sums are formed
 * on the device in integers, so the bytes depend neither on the order in which the sub-frames finish nor on the
 * number of devices.  k = 1 is exactly mtb_render_batch_ss.  The library chooses no sub-frames itself: a camera path
 * over the shutter interval gives motion blur, jittered positions on an area light give soft shadows.
 *
 * cams: n_out * subframes entries, output-major.  lights: n_out * subframes * n_lights entries, or NULL (every
 * sub-frame uses the context's lights).  rgb_out: HOST, n_out * image_h * image_w * 3 bytes, view-major.
 * subframes >= 1, n_out >= 1 and n_out * subframes <= 65535 (one grid row per sub-frame), else MTB_ERR_ARG; every
 * other argument rule is that of mtb_render_batch_ss.  stats (nullable): those of the n_out * subframes sub-frames at
 * (s*image_w) x (s*image_h) (rays and, under MTB_FLAG_COUNT_WORK, every work counter).  With several devices, device g
 * renders a contiguous range of output views with all their sub-frames; there is no gather.  There are no debug or
 * tap planes of accumulated views: mtb_render_batch_debug returns those of the sub-frames. */
int mtb_render_batch_accum(mtb_context *ctx, const mtb_camera *cams, int32_t n_out, int32_t subframes, const mtb_light *lights,
                           int32_t n_lights, int image_w, int image_h, int samples_per_axis, int max_depth, uint8_t *rgb_out,
                           mtb_stats *stats);
/* Same, returns once queued (rgb_out pinned, from mtb_host_alloc; mtb_wait joins). */
int mtb_render_batch_accum_async(mtb_context *ctx, const mtb_camera *cams, int32_t n_out, int32_t subframes,
                                 const mtb_light *lights, int32_t n_lights, int image_w, int image_h, int samples_per_axis,
                                 int max_depth, uint8_t *rgb_out);

/* Batches into DEVICE memory: every batch form above, with its outputs left in HBM of device 0 and the work ordered on
 * the caller's stream, for a consumer on the GPU (a torch model, object-id planes as segmentation masks, a second pass
 * over the hit points) that would otherwise copy the outputs to the host and upload them again.  The bytes written are
 * exactly those of the host form with the same arguments:
 *   subframes == 1, no plane:    mtb_render_batch_ss (samples_per_axis = 1: mtb_render_batch);
 *   subframes == 1, any plane:   mtb_render_batch_debug (planes on the sample grid, view-major);
 *   subframes > 1:               mtb_render_batch_accum (planes are refused, as there).
 * Argument rules, limits and the partition rule are those of the host forms; cams and lights are HOST memory and may
 * be reused as soon as the call returns.  d_rgb (n_out * image_h * image_w * 3 bytes, any alignment) must not be NULL;
 * d_dbg, d_taps and each pointer inside d_taps may be NULL.  Every output pointer must be device memory of the context's
 * device 0, d_dbg and the sig_* planes 8-byte aligned and n_rays 4-byte aligned; anything else (host memory, pageable or
 * pinned; memory of another device; misaligned planes) is MTB_ERR_ARG, before anything is queued.
 *
 * stream: a cudaStream_t of device 0 (NULL = the context's own stream).  The batch starts after all work queued on it
 * before the call, and work queued on it after the call sees the finished outputs of every device, so a caching
 * allocator (torch's) reuses an output dropped after the call only for work ordered after the batch.  stats == NULL:
 * the call returns once its work is queued, with no host synchronisation (it may still wait for its own streams when a
 * per-device buffer grows); stats != NULL: it waits for the batch and fills stats as the host forms do.  The call
 * uploads view records from host memory, so it cannot be captured into a CUDA graph: a capturing stream is
 * MTB_ERR_ARG.  With several devices, device 0 renders straight into the caller's buffers and every other device
 * renders its slice into its own and copies it over with one device-to-device copy per output, on its own stream. */
int mtb_render_batch_device(mtb_context *ctx, const mtb_camera *cams, int32_t n_out, int32_t subframes, const mtb_light *lights,
                            int32_t n_lights, int image_w, int image_h, int samples_per_axis, int max_depth, void *d_rgb,
                            mtb_debug *d_dbg, const mtb_taps *d_taps, void *stream, mtb_stats *stats);

/* Depth of field: the batch forms with a thin-lens sample per sub-frame.  With S = start_point, Dy = delta_scanline,
 * Dx = delta_pixel of the sensor of sub-frame u at (s*image_w) x (s*image_h) (mtb_camera_sensor), O its origin and
 * (u, v, f) = lenses[u], every operation in FP64 and in the order written (Cross, Dot, Normalized of the reference's
 * math3d.h), once per sub-frame:
 *     n  = Normalized(Cross(Dy, Dx));  if Dot(n, S) < 0: n = -n          focal-plane normal
 *     ex = Normalized(Dx)                                                 image right
 *     ey = Cross(n, ex);               if Dot(ey, Dy) < 0: ey = -ey        image down
 *     L  = ex * u + ey * v                                                lens point, relative to O
 * and for sample (X, Y) of its sample grid, with d = Normalized(S + Dy * Y + Dx * X) the pinhole direction:
 *     u == 0 and v == 0:   origin O,      direction d                     (the pinhole ray)
 *     otherwise:           t = f / Dot(d, n);  origin O + L,  direction Normalized(d * t - L)
 * Every ray of a sub-frame passes through the same focal plane, at distance f from O along n: that plane is in focus,
 * and the mean over sub-frames with lens points spread over an aperture blurs everything in front of it and behind
 * it.  The sample is the reference's TraceRay of that primary ray at depth max_depth (reflection, refraction, shadows
 * and quantisation unchanged), and the output bytes are those of mtb_render_batch_accum over these samples (the
 * rounded mean of the k*s*s quantised samples of an output pixel; k = 1: the sub-frame itself).  The library chooses no
 * samples: the aperture shape, the sample pattern and the focus are the caller's.
 *
 * lenses: one entry per camera (n_out * subframes), HOST memory.  Planes (dbg_out, taps) are those of
 * mtb_render_batch_debug for the lens rays and only available with subframes == 1.  Every argument rule of
 * mtb_render_batch_debug / mtb_render_batch_accum applies; in addition each of these is MTB_ERR_ARG, before anything is
 * queued: lenses == NULL (the pinhole forms are the other entry points); u, v or focus_distance not finite, or
 * focus_distance <= 0; a sub-frame whose four sample-grid corner directions c do not all satisfy Dot(n, c) > 0 (a
 * degenerate view, such as aov 0, or an aov of about 180 degrees), which also makes t finite and positive for every
 * sample.  Synchronous. */
int mtb_render_batch_lens(mtb_context *ctx, const mtb_camera *cams, const mtb_lens *lenses, int32_t n_out, int32_t subframes,
                          const mtb_light *lights, int32_t n_lights, int image_w, int image_h, int samples_per_axis, int max_depth,
                          uint8_t *rgb_out, mtb_debug *dbg_out, const mtb_taps *taps, mtb_stats *stats);
/* The same into DEVICE memory: the contract of mtb_render_batch_device (pointer and stream checks, stream ordering,
 * the split over devices) with the lens samples and rules of mtb_render_batch_lens. */
int mtb_render_batch_lens_device(mtb_context *ctx, const mtb_camera *cams, const mtb_lens *lenses, int32_t n_out, int32_t subframes,
                                 const mtb_light *lights, int32_t n_lights, int image_w, int image_h, int samples_per_axis, int max_depth,
                                 void *d_rgb, mtb_debug *d_dbg, const mtb_taps *d_taps, void *stream, mtb_stats *stats);

/* Panoramas: the batch forms with a longitude / latitude sample grid instead of the pinhole sensor, for equirectangular
 * and omni-directional stereo (ODS) views.  Each camera's origin, pitch, yaw and roll are used and its aov is ignored.
 * With Wg x Hg = (s*image_w) x (s*image_h) the sample grid, every operation in FP64 and in the order written
 * (compiled with --fmad=false / -ffp-contract=off), once per call, for column X < Wg and row Y < Hg:
 *     lon_X = ((double)(2X + 1 - Wg) / (double)(2 Wg)) * (h_fov * (M_PI / 180.0))      positive = right
 *     lat_Y = ((double)(Hg - 2Y - 1) / (double)(2 Hg)) * (v_fov * (M_PI / 180.0))      positive = up
 *     cl_X = cos(lon_X), sl_X = sin(lon_X), cp_Y = cos(lat_Y), sp_Y = sin(lat_Y)       (the C library's cos / sin)
 * once per sub-frame u, with aim = Mul(Mul(RotY(yaw), RotX(pitch)), RotZ(roll)) the rotation of mtb_camera_sensor:
 *     F = Apply(aim, (0, 0, 1)),  R = Apply(aim, (-1, 0, 0)),  U = Apply(aim, (0, 1, 0))
 * (R points along the pinhole sensor's delta_pixel and U against its delta_scanline), and per sample (X, Y), with O the
 * camera's origin and e = eye_offsets[u]:
 *     h      = F * cl_X + R * sl_X
 *     d      = Normalized(h * cp_Y + U * sp_Y)
 *     origin = O + (R * cl_X - F * sl_X) * e            (e == 0: O itself)
 * The sample is the reference's TraceRay of (origin, d) at depth max_depth, and the output bytes are those of
 * mtb_render_batch_accum over these samples (the rounded mean of the k*s*s quantised samples of an output pixel; k = 1:
 * the sub-frame itself).  h_fov = 360 and v_fov = 180 give a full equirectangular panorama whose left and right edges
 * meet without a seam; e = -IPD/2 and +IPD/2 give the left and right eye of an ODS pair, the eye displaced along each
 * column's tangent.  The library chooses no field of view, eye distance or sample pattern.  mtb_panorama_rays returns
 * the rays of one sub-frame.
 *
 * eye_offsets: NULL (all 0) or one entry per camera (n_out * subframes), HOST memory.  Planes (dbg_out, taps) are those
 * of mtb_render_batch_debug for the panorama rays and only available with subframes == 1.  Every argument rule of
 * mtb_render_batch_debug / mtb_render_batch_accum applies; in addition each of these is MTB_ERR_ARG, before anything is
 * queued (also on a host-only context): h_fov not finite or outside (0, 360]; v_fov not finite or outside (0, 180]; an
 * eye offset that is not finite.  Synchronous. */
int mtb_render_batch_pano(mtb_context *ctx, const mtb_camera *cams, const double *eye_offsets, int32_t n_out, int32_t subframes, double h_fov,
                          double v_fov, const mtb_light *lights, int32_t n_lights, int image_w, int image_h, int samples_per_axis, int max_depth,
                          uint8_t *rgb_out, mtb_debug *dbg_out, const mtb_taps *taps, mtb_stats *stats);
/* The same into DEVICE memory: the contract of mtb_render_batch_device (pointer and stream checks, stream ordering,
 * the split over devices) with the panorama arguments and rules of mtb_render_batch_pano. */
int mtb_render_batch_pano_device(mtb_context *ctx, const mtb_camera *cams, const double *eye_offsets, int32_t n_out, int32_t subframes,
                                 double h_fov, double v_fov, const mtb_light *lights, int32_t n_lights, int image_w, int image_h,
                                 int samples_per_axis, int max_depth, void *d_rgb, mtb_debug *d_dbg, const mtb_taps *d_taps, void *stream,
                                 mtb_stats *stats);

/* Same render, result left in DEVICE memory of device 0 (d_rgb: chunk_w*chunk_h*3 bytes); enqueued on
 * `stream` (a cudaStream_t of device 0; NULL = the context's own stream) without synchronising when the
 * context has one device.  This is the entry bench.py times for the HBM-resident figure. */
int mtb_render_chunk_device(mtb_context *ctx, const mtb_camera *cam, int image_w, int image_h, int chunk_x,
                            int chunk_y, int chunk_w, int chunk_h, int max_depth, void *d_rgb, void *stream,
                            mtb_stats *stats);

/* Frames shared between processes - the in-box form of the master's frame that workers blit into
 * (main_net_master.cc:223-236) when every GPU is driven by its own process.  The gathering process creates the frame
 * on its device and passes the 64-byte handle to the others by any means (bench.py: torch.distributed broadcast);
 * they open it and hand the mapped pointer to mtb_render_chunk_device as d_rgb: with mtb_set_partition in effect
 * their kernels then store the tiles they own straight into the gatherer's HBM over NVLink (cudaIpc* peer mapping),
 * and the frame is complete when every process has finished its call - no gather copy, no collective on the data
 * path.  mtb_frame_release frees (creator) or unmaps (opener) the frame; mtb_destroy releases what is left. */
#define MTB_FRAME_HANDLE_BYTES 64
int mtb_frame_create(mtb_context *ctx, size_t bytes, void **d_ptr, unsigned char handle[MTB_FRAME_HANDLE_BYTES]);
int mtb_frame_open(mtb_context *ctx, const unsigned char handle[MTB_FRAME_HANDLE_BYTES], void **d_ptr);
int mtb_frame_release(mtb_context *ctx, void *d_ptr);
/* Waits for the context's devices, then copies `bytes` bytes at `offset` of a frame to host memory. */
int mtb_frame_read(mtb_context *ctx, const void *d_ptr, size_t offset, size_t bytes, void *host_out);

/* Work counters accumulated by mtb_render_chunk_device calls that passed stats == NULL since the last
 * read; synchronises every device of the context and resets the counters. */
int mtb_read_counters(mtb_context *ctx, mtb_stats *stats);

/* Pipeline in use on device 0: 0 = megakernel, 3 = queue pipeline, -1 = still measuring (codes 1 and 2 belonged to
 * retired pipelines); the timed megakernel / queue-pipeline frames (ms) of the automatic choice are returned when the
 * pointers are non-NULL. */
int mtb_pipeline_in_use(const mtb_context *ctx, float *mega_ms, float *wavefront_ms);
/* Retired with hybrid frames: always 0.0f.  Kept so that callers built against earlier versions still link. */
float mtb_hybrid_share(const mtb_context *ctx);
/* Number of kernels of this library launched on this context so far (bench.py's gpu_launches). */
uint64_t mtb_launch_count(const mtb_context *ctx);

/* Batched OctTree::IntersectRay (octtree.cc:26-40).  HOST arrays: origins/dirs n*3, tri_index n (insertion
 * index, -1 = nullptr), t n, point n*3 (nullable).  Miss contract: tri_index[i] = -1, t[i] = NaN, point[i] = NaN
 * (the reference leaves its out-parameters untouched on a miss, octtree.cc:36-39; a batched call writes whole
 * arrays, so the untouched state is spelled NaN).  The C++ shim's single-ray IntersectRay leaves *point and
 * *distance untouched on a miss like the reference. */
int mtb_intersect_rays(mtb_context *ctx, int64_t n, const double *origins, const double *dirs, int32_t *tri_index,
                       double *t, double *point, mtb_stats *stats);

/* Camera::GetSensor (camera.cc:17-63): start_point, delta_scanline, delta_pixel (9 doubles), host side. */
int mtb_camera_sensor(const mtb_camera *cam, int image_w, int image_h, double out9[9]);

/* The primary rays of one panorama sub-frame of mtb_render_batch_pano (its contract, bit for bit) on a grid_w x grid_h
 * sample grid, host side: origins (nullable) and dirs are grid_h * grid_w * 3 doubles, row-major, sample (X, Y) at
 * (Y * grid_w + X) * 3.  MTB_ERR_ARG for a NULL cam or dirs, a grid side outside 1..65536, and the h_fov, v_fov and
 * eye_offset rules of mtb_render_batch_pano.  Needs no context and no device. */
int mtb_panorama_rays(const mtb_camera *cam, int grid_w, int grid_h, double h_fov, double v_fov, double eye_offset, double *origins,
                      double *dirs);

const char *mtb_version(void);

#ifdef __cplusplus
}
#endif
#endif /* MYTHTRACER_B200_H_ */
