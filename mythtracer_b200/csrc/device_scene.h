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
  // Repair launch: the wavefront pipeline runs without reading anything back to the host; if its activation table
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

// Accumulated batch (LaunchRenderMegaBatch with subframes k > 1): grid row u is sub-frame u of output view u / k.
// Both arrays cover the output views of the launch and are zero when it starts.
struct AccumParams {
  uint32_t *sum;       // per output view: W x H x 3 sums of the k * s * s quantised samples of each output channel
  uint32_t *arrive;    // per output view, tile of the sample grid and warp half: warps that have added their sums
  int32_t subframes;   // k; 1: no accumulation (sum and arrive unused)
};

// Thin-lens sample of one grid row (sub-frame) of a batch launch, from mtb_lens on the host (RenderBatchImpl).  The
// primary ray of sample (X, Y), with d the pinhole direction of that sample and O the view's origin, starts at O + shift
// and points along Normalized(d * (focus / Dot(d, axis)) - shift).  centred != 0 (u = v = 0): the pinhole ray itself.
struct LensRec {
  double shift[3];  // L: the lens point relative to O
  double axis[3];   // n: unit normal of the focal plane, facing the sensor
  double focus;     // focus_distance along n
  uint32_t centred;
};

// Panorama of one grid row (sub-frame) of a batch launch, from the camera and eye offset on the host
// (RenderBatchImpl).  With {cl, sl} = lon[X] and {cp, sp} = lat[Y], sample (X, Y) is traced along
// Normalized((forward * cl + right * sl) * cp + up * sp) from O, or from O + (right * cl - forward * sl) * eye when
// eye != 0 (O the view's origin).
struct PanoRec {
  double forward[3], right[3], up[3];  // the camera's basis (ComputePanoramaBasis)
  double eye;                          // e: the offset along the column's tangent
};

// The panorama of a batch launch: one PanoRec per grid row, and the {cos, sin} tables of the sample grid's longitudes
// (one per column) and latitudes (one per row), each entry 16-byte aligned.  rec == NULL: no panorama.
struct PanoParams {
  const PanoRec *rec;
  const double *lon, *lat;
};

struct IntersectParams {
  int64_t n;
  const double *origins, *dirs;
  int32_t *tri_index;
  double *t, *point;
  unsigned long long *counters;
};

// Buffers of the wavefront pipeline (wavefront.cu), all resident in HBM.  An activation is one TraceRayWorker call
// (mythtracer.cc:13): a primary ray, or a reflection / refraction child of an earlier activation.  ONE ray queue holds
// every level, entry id = activation id, and ids [0, P) are the pixel slots.  A queued ray lives in act_point (origin)
// / act_dir (direction) / act_coef / act_path / act_pixel / act_info (level | in_object << 8) of its activation until
// a warp takes it; act_ready[id] == epoch of the frame once the entry is complete.
struct WfBuffers {
  int32_t *act_mtl;    // material index of the hit; < 0: nothing to light (miss or mtl == nullptr)
  double *act_point, *act_dir;  // 3 doubles each
  int32_t *act_pixel;  // chunk-local pixel (taps)
  unsigned long long *act_path;  // path code (1 = root, 2p = reflection child, 2p+1 = refraction child)
  double *act_color;   // 3 doubles: local colour, later the folded colour
  int32_t *act_refl, *act_refr;  // child activation ids (-1: none)
  // Device-side frame control (nothing of it is read by the host while a frame is in flight):
  uint32_t *ctrl;      // [0] overflow flag (the table was too small: the frame is rendered by the repair launch)
  unsigned long long *work;  // [kNumCounters] work counters of this frame, committed by WfCommit unless it overflowed
  int32_t act_cap;
  double *act_coef;
  int32_t *act_info;
  uint32_t *act_ready;
  uint32_t *qctl;  // [kQHead] next entry to hand out, [kQTail] entries reserved, [kQPending] activations not finished yet
  // Unused.  With a parameter block 16 bytes smaller, ptxas keeps more of WfQueue's parameters in registers and spills
  // more (218 -> 250 B of spill stores): measured on a B200 at 1000 W, C3 through the queue pipeline took 9.75 ms
  // instead of 9.28 ms, C4 7.5 instead of 7.2 ms.
  uint64_t reserved[2];
};
enum QueueCtl { kQHead = 0, kQTail = 1, kQPending = 2, kQWords = 4 };
// layout of the pinned host copy WfCommit writes: overflow flag, frame sequence
constexpr int kWfHostOverflow = 0;
constexpr int kWfHostSequence = 1;
constexpr int kWfHostWords = 2;

// wavefront.cu: one persistent kernel for all levels (WfQueue), then the per-pixel fold + V3DtoRGB (WfResolveTree).
void LaunchWfQueueBegin(const WfBuffers &wf, int slots, cudaStream_t stream);
void LaunchWfQueue(const DeviceScene &sc, const RenderParams &rp, const WfBuffers &wf, int slots, unsigned epoch, int sm_count, bool debug_build,
                   cudaStream_t stream);
void LaunchWfResolveTree(const DeviceScene &sc, const RenderParams &rp, const WfBuffers &wf, int slots, cudaStream_t stream);
void LaunchWfCommit(const WfBuffers &wf, unsigned long long *global, uint32_t *host_copy, cudaStream_t stream);

// megakernel.cu
// Builds tile_order (descending cost, bucketed) from tile_cost and clears tile_cost for the coming frame.
void LaunchBuildTileOrder(uint32_t *tile_cost, int32_t *tile_order, int n_tiles, cudaStream_t stream);
// One 8x8 tile per 64-thread block; n_blocks = tiles of the launch (rp.tiles_x in units of 8 pixels).
void LaunchRenderMega(const DeviceScene &sc, const RenderParams &rp, int n_blocks, bool debug_build, cudaStream_t stream);
// n_views whole frames in one launch: grid (tiles_per_view, n_views), camera of view v = views[v] (device memory), its
// lights sc.lights + v * sc.n_lights, its pixels rp.rgb + v * chunk_w * chunk_h * 3, its debug / tap entries (each
// plane nullable) rp.dbg / sig_hits / sig_shadow / n_rays + v * chunk_w * chunk_h.  rp.strip_first = 0,
// rp.strip_stride = 1, and tile_order / tile_cost / run_if NULL.
// samples_per_axis s = 2, 4 or 8: supersampled views.  rp.chunk_w x rp.chunk_h (and views[v].sensor) describe the
// s*W x s*H sample grid, tiles_per_view counts its tiles, and view v's W x H output pixels (each the rounded mean of
// its s x s samples) go to rp.rgb + v * W * H * 3.  s = 1: the plain batch above.
// acc.subframes k > 1: accumulated views.  n_views counts sub-frames (a multiple of k); sub-frame u is traced exactly as
// view u above, and output view v = u / k (W x H, at rp.rgb + v * W * H * 3) is the rounded mean of the k * s * s
// samples of its sub-frames, summed in acc.sum (zeroed by the caller, with acc.arrive, before the launch).  The planes
// must be NULL.  k = 1: the batches above.
// lens (device memory, nullable): one LensRec per grid row (sub-frame); the primary rays of row u are those of lens[u].
// NULL: pinhole views, the kernels above.
// pano.rec (device memory, nullable, never with lens): panoramas; the primary rays of row u are those of pano.rec[u] and
// the launch's longitude / latitude tables (views[u].sensor is unused).  NULL: the kernels above.
void LaunchRenderMegaBatch(const DeviceScene &sc, const RenderParams &rp, const ViewRec *views, int tiles_per_view, int n_views,
                           int samples_per_axis, const AccumParams &acc, const LensRec *lens, const PanoParams &pano, bool debug_build,
                           cudaStream_t stream);
void LaunchIntersect(const DeviceScene &sc, const IntersectParams &ip, bool debug_build, cudaStream_t stream);  // one ray per thread

}  // namespace mtb
