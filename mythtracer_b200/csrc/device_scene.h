// Structures shared by the host API (api.cu) and the kernels (megakernel.cu, wavefront.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "mythtracer_b200.h"
#include "scene_build.h"

namespace mtb {

// Everything the kernels read, resident in the HBM of one device.
struct DeviceScene {
  const NodeRec *nodes;
  const SlotRec *slots;
  const ShadeRec *shade;
  const BvhRec *bvh;
  const int32_t *list_order;
  const int32_t *slot_node;  // canonical slot -> octree node holding it
  const Bvh2Node *gnodes;   // scene BVH of the certified fast traversal; NULL: exact octree recursion only
  const SlotRec *gslots;    // the triangles in scene-BVH leaf order (SlotRec::canon = slot in slots / shade)
  const mtb_material *materials;
  cudaTextureObject_t tex_atlas;  // ONE point-sampled layered texture object: layer = texture index, one RGBA32 texel per 32-bit word
  const int2 *texture_dim;
  const mtb_light *lights;
  int32_t n_lights;
  int32_t n_materials;
  int32_t n_nodes;
  // FP32 list-BVH cull: largest |coordinate| of the scene box; 0 disables the FP32 path (boxes are then
  // evaluated in FP64, still conservatively)
  float cull_radius;
  // largest extent of any triangle's box along any axis (bounds |e1|, |e2| in the error model of LimitPrune)
  float max_tri_extent;
};

// Work counters, one slot per field of mtb_stats' integer part (same order).
enum Counter {
  kRays = 0, kPrimary, kShadow, kReflect, kRefract, kSlab, kVisit, kTriAabb, kMt, kHit, kShade, kBvh, kLiteral, kFast, kFallback,
  kLongRays128, kLongVisits128, kLongRays512, kLongVisits512,
  kNumCounters
};

struct RenderParams {
  double sensor[9];   // start_point, delta_scanline, delta_pixel (camera.cc:56-62)
  double origin[3];
  int32_t image_w, image_h;
  int32_t chunk_x, chunk_y, chunk_w, chunk_h;
  int32_t max_depth;
  // The chunk is cut into strips of 8 rows; this launch renders strips strip_first + i * strip_stride
  // (multi-GPU / multi-process interleave).  Block b <-> 8x8 tile (b % tiles_x) of local strip b / tiles_x.
  int32_t tiles_x, strip_first, strip_stride;
  uint8_t *rgb;        // chunk-local RGB24, stride chunk_w*3 (may be peer memory of device 0)
  mtb_debug *dbg;      // nullable
  uint64_t *sig_hits;  // nullable taps
  uint64_t *sig_shadow;
  uint32_t *n_rays;
  unsigned long long *counters;  // kNumCounters, nullable unless the counting build runs
  // Cost-aware tile scheduling of the megakernel: block b renders tile tile_order[b] (NULL: b) and adds the
  // rays it traced to tile_cost[tile]; the next frame launches the most expensive tiles first.
  const int32_t *tile_order;
  uint32_t *tile_cost;
  // Hybrid frame: the first *heavy_k tiles of tile_order (the most expensive ones of the previous frame) are
  // rendered by the wavefront pipeline, the rest by the megakernel, concurrently.  NULL: no split.
  const int32_t *heavy_k;
  // Which side of the split a RenderMega launch renders: 0 = positions >= *heavy_k (the megakernel half of a hybrid
  // frame; everything when heavy_k is NULL), 1 = positions < *heavy_k (the wavefront's tiles: the repair launch below).
  int32_t mega_part;
  // Repair launch: the wavefront pipeline runs without reading anything back to the host; if one of its queues
  // overflowed, *run_if != 0 and a RenderMega launch queued behind it renders the wavefront's tiles again (both
  // pipelines produce the same bytes).  NULL: unconditional launch.  Blocks of a launch with *run_if == 0 exit at once.
  const uint32_t *run_if;
};

// One view of a batch launch (LaunchRenderMegaBatch): its camera as Camera::GetSensor leaves it (ComputeSensor on the
// host).  The lights of view v are DeviceScene::lights[v * n_lights ..] of the scene copy the batch launch passes.
struct ViewRec {
  double sensor[9];  // start_point, delta_scanline, delta_pixel
  double origin[3];
};

struct IntersectParams {
  int64_t n;
  const double *origins, *dirs;
  int32_t *tri_index;
  double *t, *point;
  unsigned long long *counters;
};

// Buffers of the wavefront pipeline (wavefront.cu), all resident in HBM.  A "level" is one generation of
// TraceRayWorker activations (mythtracer.cc:13): level 0 = primary rays, level L+1 = the reflection and
// refraction children of level L.  Activations are numbered level by level, so activation id =
// act_base(level) + position in the level's queue, and ids [0, P) are the pixels.
struct WfBuffers {
  // ray queues, ping-pong by level parity: origin, direction (3 doubles each), current_reflection_coef,
  // path code (1 = root, 2p = reflection child, 2p+1 = refraction child), chunk-local pixel, in_object
  double *rq_o[2], *rq_d[2], *rq_coef[2];
  unsigned long long *rq_path[2];
  int32_t *rq_pixel[2];
  unsigned char *rq_inobj[2];
  // activation table, indexed by activation id.  Shading context written by WfTraceMain and read by the
  // shadow / light kernels, which run on a second stream concurrently with the deeper levels' traces:
  int32_t *act_mtl;    // material index of the hit; < 0: nothing to light (miss or mtl == nullptr)
  double *act_point, *act_normal, *act_surface, *act_reflected, *act_dir;  // 3 doubles each
  int32_t *act_pixel;  // chunk-local pixel (taps)
  unsigned long long *act_path;
  double *sh_power;    // [light][activation][3]  light_power after the shadow walk
  uint32_t *sh_flags;  // [light][activation]     in_shadow | segments << 1
  double *act_color;   // 3 doubles: local colour, later the folded colour
  int32_t *act_refl, *act_refr;  // child activation ids (-1: none)
  // Device-side frame control (nothing of it is read by the host while a frame is in flight):
  uint32_t *level_n;   // [MTB_MAX_RAY_DEPTH + 2] rays queued per level; [0] = pixel slots
  uint32_t *ctrl;      // [0] overflow flag (a queue was too small: the frame is rendered by the repair launch)
  unsigned long long *work;  // [kNumCounters] work counters of this frame, committed by WfCommit unless it overflowed
  int32_t queue_cap, act_cap;
  // Queue pipeline (WfQueue): ONE ray queue for all levels, entry id = activation id.  A queued ray lives in
  // act_point (origin) / act_dir (direction) / act_coef / act_path / act_pixel / act_info (level | in_object << 8)
  // of its activation until a warp takes it; act_ready[id] == epoch of the frame once the entry is complete.
  double *act_coef;
  int32_t *act_info;
  uint32_t *act_ready;
  uint32_t *qctl;  // [kQHead] next entry to hand out, [kQTail] entries reserved, [kQPending] activations not finished yet
};
enum QueueCtl { kQHead = 0, kQTail = 1, kQPending = 2, kQWords = 4 };
// layout of the pinned host copy WfCommit writes: level_n[0 .. MTB_MAX_RAY_DEPTH + 1], overflow flag, frame sequence
constexpr int kWfHostOverflow = MTB_MAX_RAY_DEPTH + 2;
constexpr int kWfHostSequence = MTB_MAX_RAY_DEPTH + 3;
constexpr int kWfHostWords = MTB_MAX_RAY_DEPTH + 4;

// wavefront.cu.  `expect` = rays the level is expected to hold (sizes the grid only; the kernels read the real count
// on the device and loop grid-strided).
void LaunchWfBegin(const WfBuffers &wf, int slots, cudaStream_t stream);
void LaunchWfTrace(const DeviceScene &sc, const RenderParams &rp, const WfBuffers &wf, int level, long long expect, bool debug_build,
                   cudaStream_t stream);
void LaunchWfShadow(const DeviceScene &sc, const RenderParams &rp, const WfBuffers &wf, int level, long long expect, bool debug_build,
                    cudaStream_t stream);
void LaunchWfLight(const DeviceScene &sc, const RenderParams &rp, const WfBuffers &wf, int level, long long expect, cudaStream_t stream);
void LaunchWfFold(const DeviceScene &sc, const WfBuffers &wf, int level, long long expect, cudaStream_t stream);
void LaunchWfResolve(const RenderParams &rp, const WfBuffers &wf, int n_slots, cudaStream_t stream);
void LaunchWfCommit(const WfBuffers &wf, unsigned long long *global, uint32_t *host_copy, cudaStream_t stream);
// Queue pipeline: one persistent kernel for all levels (WfQueue), then the per-pixel fold + V3DtoRGB (WfResolveTree).
void LaunchWfQueueBegin(const WfBuffers &wf, int slots, cudaStream_t stream);
void LaunchWfQueue(const DeviceScene &sc, const RenderParams &rp, const WfBuffers &wf, int slots, unsigned epoch, int sm_count, bool debug_build,
                   cudaStream_t stream);
void LaunchWfResolveTree(const DeviceScene &sc, const RenderParams &rp, const WfBuffers &wf, int slots, cudaStream_t stream);

// megakernel.cu
// Builds tile_order (descending cost, bucketed) from tile_cost and clears tile_cost for the coming frame.
// heavy_k (nullable): receives the number of leading tiles of the order that carry heavy_share_q16 / 65536 of the
// frame's rays (at most k_max tiles).
void LaunchBuildTileOrder(uint32_t *tile_cost, int32_t *tile_order, int n_tiles, int32_t *heavy_k, int k_max, unsigned heavy_share_q16,
                          cudaStream_t stream);
// One 8x8 tile per 64-thread block; n_blocks = tiles of the launch (rp.tiles_x in units of 8 pixels).
void LaunchRenderMega(const DeviceScene &sc, const RenderParams &rp, int n_blocks, bool debug_build, cudaStream_t stream);
// n_views whole frames in one launch: grid (tiles_per_view, n_views), camera of view v = views[v] (device memory), its
// lights sc.lights + v * sc.n_lights, its pixels rp.rgb + v * chunk_w * chunk_h * 3.  rp.strip_first = 0,
// rp.strip_stride = 1, and tile_order / tile_cost / heavy_k / run_if / taps / dbg NULL.
// samples_per_axis s = 2, 4 or 8: supersampled views.  rp.chunk_w x rp.chunk_h (and views[v].sensor) describe the
// s*W x s*H sample grid, tiles_per_view counts its tiles, and view v's W x H output pixels (each the rounded mean of
// its s x s samples) go to rp.rgb + v * W * H * 3.  s = 1: the plain batch above.
void LaunchRenderMegaBatch(const DeviceScene &sc, const RenderParams &rp, const ViewRec *views, int tiles_per_view, int n_views,
                           int samples_per_axis, bool debug_build, cudaStream_t stream);
void LaunchIntersect(const DeviceScene &sc, const IntersectParams &ip, bool debug_build, int mode, cudaStream_t stream);  // mode 0: one ray per thread, 1: two rays per lane (Trace2), 2: chain (TraceChain), 3: two calls

}  // namespace mtb
