// C ABI of mythtracer_b200 (see include/mythtracer_b200.h): context, scene residency in HBM, and the
// launch / gather logic around the kernels of megakernel.cu / wavefront.cu.  No CPU rendering path exists in this file.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "device_scene.h"

namespace mtb {
// device_build.cu
cudaError_t BuildSceneBvhOnDevice(const double *h_ref_box, int64_t n_refs, const double scene_box[6], double pad, cudaStream_t stream,
                                  Bvh2Node **d_nodes_out, int32_t *n_nodes_out, int32_t **d_leaf_ref_out, int32_t *depth_out);
void LaunchGatherLeafSlots(const SlotRec *slots, const int32_t *ref_slot, const int32_t *leaf_ref, int64_t n_positions, SlotRec *gslots,
                           cudaStream_t stream);
}  // namespace mtb

namespace {

std::string g_create_error;

// (the devices of a context are driven by one host thread each while a frame is in flight, hence the lock)
#define MTB_CUDA(ctx, expr)                                                                                  \
  do {                                                                                                       \
    cudaError_t e__ = (expr);                                                                                \
    if (e__ != cudaSuccess) {                                                                                \
      std::lock_guard<std::mutex> lock__((ctx)->err_mutex);                                                  \
      (ctx)->err = std::string(#expr) + ": " + cudaGetErrorString(e__);                                      \
      return MTB_ERR_CUDA;                                                                                   \
    }                                                                                                        \
  } while (0)

template <typename T>
struct DeviceBuffer {
  T *ptr = nullptr;
  size_t count = 0;
  cudaError_t Reserve(size_t n) {
    if (n <= count && ptr != nullptr) return cudaSuccess;
    if (ptr != nullptr) cudaFree(ptr);
    ptr = nullptr;
    count = 0;
    if (n == 0) return cudaSuccess;
    cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&ptr), n * sizeof(T));
    if (e == cudaSuccess) count = n;
    return e;
  }
  cudaError_t Upload(const T *src, size_t n, cudaStream_t s) {
    cudaError_t e = Reserve(n > 0 ? n : 1);
    if (e != cudaSuccess || n == 0) return e;
    return cudaMemcpyAsync(ptr, src, n * sizeof(T), cudaMemcpyHostToDevice, s);
  }
  void Free() {
    if (ptr != nullptr) cudaFree(ptr);
    ptr = nullptr;
    count = 0;
  }
};

struct DeviceState {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev_start = nullptr, ev_stop = nullptr;
  cudaEvent_t ev_gathered = nullptr;  // device 0 only: the last gather has read every peer buffer
  cudaStream_t l2_window_stream = nullptr;  // stream that carries the L2 access-policy window (MTB_L2_PERSIST_MB)
  bool peer_to_dev0 = false;     // device 0 can read this device's memory (peer-copy gather)
  bool peer_store_dev0 = false;  // this device's kernels can store into device 0's memory (direct tile stores)
  // scene
  DeviceBuffer<mtb::NodeRec> nodes;
  DeviceBuffer<mtb::SlotRec> slots;
  DeviceBuffer<mtb::ShadeRec> shade;
  DeviceBuffer<mtb::BvhRec> bvh;
  DeviceBuffer<mtb::Bvh2Node> gnodes;   // scene BVH of the certified fast traversal
  DeviceBuffer<mtb::SlotRec> gslots;
  DeviceBuffer<int32_t> list_order;
  DeviceBuffer<int32_t> slot_node;
  DeviceBuffer<int32_t> leaf_ref, ref_slot;  // device-built scene BVH: leaf position -> reference -> canonical slot
  int32_t device_bvh_depth = 0;
  DeviceBuffer<mtb_material> materials;
  DeviceBuffer<int2> tex_dims;
  DeviceBuffer<mtb_light> lights;
  std::vector<cudaArray_t> tex_arrays;
  std::vector<cudaTextureObject_t> tex_handles;
  mtb::DeviceScene scene{};
  // per-render scratch
  DeviceBuffer<uint8_t> rgb;
  DeviceBuffer<mtb_debug> dbg;
  DeviceBuffer<uint64_t> sig_hits, sig_shadow;
  DeviceBuffer<uint32_t> n_rays;
  DeviceBuffer<unsigned long long> counters;
  // cost-aware tile order of the megakernel (previous frame's per-tile ray counts)
  DeviceBuffer<uint32_t> tile_cost;
  DeviceBuffer<int32_t> tile_order;
  long long tile_signature = -1;  // geometry the costs were recorded for
  // run-time choice between the two pipelines (flags without a pipeline bit): both are timed once per
  // geometry (megakernel with a warm tile order, then wavefront) and the faster one is kept
  long long tune_signature = -1;
  int tune_stage = 0;           // see RenderImpl
  float tune_ms[3] = {0.f, 0.f, 0.f};  // megakernel, wavefront, hybrid
  int tune_choice = 0;                 // 0 megakernel, 1 wavefront, 2 hybrid
  // hybrid frames: the most expensive tiles go through the wavefront while the megakernel renders the rest
  DeviceBuffer<int32_t> heavy_k;
  cudaStream_t hybrid_stream = nullptr;
  cudaEvent_t ev_split = nullptr, ev_mega_done = nullptr, ev_wf_done = nullptr;  // (timed: they steer the split)
  float hybrid_share = 0.30f;     // share of the frame's rays that goes through the wavefront; steered frame by frame
  bool hybrid_timed = false;      // the three events above were recorded by the previous hybrid frame
  // batch launches (RenderBatchImpl): view records, per-view lights and the views' frames of this device, and the
  // events that time them (the single-frame events steer the automatic pipeline choice and are left alone)
  DeviceBuffer<mtb::ViewRec> batch_views;
  DeviceBuffer<mtb_light> batch_lights;
  DeviceBuffer<uint8_t> batch_rgb;
  cudaEvent_t ev_batch_start = nullptr, ev_batch_stop = nullptr;
  // intersect scratch
  DeviceBuffer<double> q_origins, q_dirs, q_t, q_point;
  DeviceBuffer<int32_t> q_tri;
  // wavefront pipeline state (wavefront.cu)
  DeviceBuffer<double> wf_rq_o[2], wf_rq_d[2], wf_rq_coef[2];
  DeviceBuffer<unsigned long long> wf_rq_path[2];
  DeviceBuffer<int32_t> wf_rq_pixel[2];
  DeviceBuffer<unsigned char> wf_rq_inobj[2];
  DeviceBuffer<double> wf_act_point, wf_act_normal, wf_act_surface, wf_act_reflected, wf_act_dir, wf_sh_power;
  DeviceBuffer<uint32_t> wf_sh_flags;
  DeviceBuffer<double> wf_act_color;
  DeviceBuffer<int32_t> wf_act_refl, wf_act_refr, wf_act_mtl, wf_act_pixel;
  DeviceBuffer<unsigned long long> wf_act_path;
  cudaStream_t wf_stream2 = nullptr;             // shadow / light kernels (side stream 0)
  cudaStream_t wf_side[3] = {nullptr, nullptr, nullptr};  // further side streams: the shadow kernels of different levels are independent
  cudaEvent_t wf_ev_side[4] = {nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t wf_ev_level[MTB_MAX_RAY_DEPTH + 2] = {};  // level L traced (main stream)
  cudaEvent_t wf_ev_lit = nullptr;               // all lights folded (second stream)
  DeviceBuffer<uint32_t> wf_level_n, wf_ctrl;
  DeviceBuffer<double> wf_act_coef;       // queue pipeline (WfQueue)
  DeviceBuffer<int32_t> wf_act_info;
  DeviceBuffer<uint32_t> wf_act_ready, wf_qctl;
  uint32_t wf_epoch = 0;                  // frame number of the queue pipeline: act_ready[id] == epoch marks a complete entry
  DeviceBuffer<unsigned long long> wf_work;
  // pinned; written by WfCommit at the end of every frame (level counts, overflow flag, frame sequence number) and read
  // by the host at the START of the next frame only: grid sizes and queue capacities follow the scene with one frame
  // of delay and without a single host read-back while a frame is in flight
  uint32_t *wf_host = nullptr;
  uint32_t wf_seen_sequence = 0;
  int wf_queue_factor = 2, wf_act_factor = 6;  // capacities in units of the pixel-slot count; doubled after an overflow
  mtb::WfBuffers wf{};

  void FreeAll() {
    nodes.Free(); slots.Free(); shade.Free(); bvh.Free(); gnodes.Free(); gslots.Free(); list_order.Free(); slot_node.Free(); leaf_ref.Free(); ref_slot.Free(); materials.Free();
    tex_dims.Free(); lights.Free(); rgb.Free(); dbg.Free(); sig_hits.Free(); sig_shadow.Free(); n_rays.Free();
    counters.Free(); tile_cost.Free(); tile_order.Free(); heavy_k.Free();
    batch_views.Free(); batch_lights.Free(); batch_rgb.Free();
    if (ev_batch_start != nullptr) cudaEventDestroy(ev_batch_start);
    if (ev_batch_stop != nullptr) cudaEventDestroy(ev_batch_stop);
    ev_batch_start = ev_batch_stop = nullptr;
    if (hybrid_stream != nullptr) cudaStreamDestroy(hybrid_stream);
    hybrid_stream = nullptr;
    if (ev_split != nullptr) cudaEventDestroy(ev_split);
    if (ev_mega_done != nullptr) cudaEventDestroy(ev_mega_done);
    if (ev_wf_done != nullptr) cudaEventDestroy(ev_wf_done);
    ev_split = ev_mega_done = ev_wf_done = nullptr; q_origins.Free(); q_dirs.Free(); q_t.Free(); q_point.Free(); q_tri.Free();
    for (int k = 0; k < 2; k++) {
      wf_rq_o[k].Free(); wf_rq_d[k].Free(); wf_rq_coef[k].Free(); wf_rq_path[k].Free(); wf_rq_pixel[k].Free();
      wf_rq_inobj[k].Free();
    }
    wf_act_point.Free(); wf_act_normal.Free(); wf_act_surface.Free(); wf_act_reflected.Free(); wf_act_dir.Free();
    wf_sh_power.Free(); wf_sh_flags.Free(); wf_act_color.Free(); wf_act_refl.Free(); wf_act_refr.Free();
    wf_act_mtl.Free(); wf_act_pixel.Free(); wf_act_path.Free(); wf_level_n.Free(); wf_ctrl.Free(); wf_work.Free(); wf_act_coef.Free(); wf_act_info.Free(); wf_act_ready.Free(); wf_qctl.Free();
    if (wf_stream2 != nullptr) cudaStreamDestroy(wf_stream2);
    wf_stream2 = nullptr;
    for (cudaStream_t &st : wf_side) {
      if (st != nullptr) cudaStreamDestroy(st);
      st = nullptr;
    }
    for (cudaEvent_t &e : wf_ev_side) {
      if (e != nullptr) cudaEventDestroy(e);
      e = nullptr;
    }
    for (cudaEvent_t &e : wf_ev_level) {
      if (e != nullptr) cudaEventDestroy(e);
      e = nullptr;
    }
    if (wf_ev_lit != nullptr) cudaEventDestroy(wf_ev_lit);
    wf_ev_lit = nullptr;
    if (wf_host != nullptr) cudaFreeHost(wf_host);
    wf_host = nullptr;
  }
};

}  // namespace

struct mtb_context {
  std::vector<DeviceState> dev;
  std::string err;
  uint32_t flags = 0;
  bool has_scene = false;
  int part_index = 0, part_count = 1;
  mtb::FlatScene flat;
  std::vector<mtb_triangle> triangles;
  std::vector<mtb_material> materials;
  std::vector<mtb::LoadedTexture> textures;
  std::vector<std::string> material_names, texture_names;
  std::vector<mtb_light> lights;
  int64_t device_bytes = 0;
  std::atomic<uint64_t> launches{0};  // kernels of this library launched so far (mtb_launch_count)
  bool no_peer_store = false;         // MTB_NO_PEER_STORE=1: gather with peer copies instead of direct tile stores (A/B)
  bool no_host_store = false;         // MTB_NO_HOST_STORE=1: copy the frame to a pinned host buffer instead of storing tiles into it (A/B)
  int l2_persist_mb = 0;              // MTB_L2_PERSIST_MB=n: pin the scene BVH's nodes in n MB of persisting L2 (A/B)
  bool device_bvh = false;            // the scene BVH of the current scene was built on the devices (device_build.cu)
  int64_t atlas_bytes = 0;            // layered texture array as allocated on a device
  double ms_parse = 0.0, ms_upload = 0.0, ms_device_bvh = 0.0;  // stages of the last load (mtb_load_timing)
  std::vector<void *> owned_frames, opened_frames;  // mtb_frame_create / mtb_frame_open
  std::mutex err_mutex;
};

namespace {

void DestroyTextures(DeviceState *d) {
  for (cudaTextureObject_t t : d->tex_handles) cudaDestroyTextureObject(t);
  for (cudaArray_t a : d->tex_arrays) cudaFreeArray(a);
  d->tex_handles.clear();
  d->tex_arrays.clear();
}

// Regular rays take the certified fast traversal over the scene BVH unless the exact octree recursion is forced.
void SelectTraversal(mtb_context *ctx, DeviceState *d) {
  const bool fast = (ctx->flags & (MTB_FLAG_EXACT_OCTREE | MTB_FLAG_NO_LIST_BVH)) == 0 && d->gnodes.ptr != nullptr && d->gnodes.count > 0 &&
                    d->gslots.ptr != nullptr && d->scene.cull_radius > 0.0f;
  d->scene.gnodes = fast ? d->gnodes.ptr : nullptr;
  d->scene.gslots = fast ? d->gslots.ptr : nullptr;
}

int UploadToDevice(mtb_context *ctx, DeviceState *d) {
  MTB_CUDA(ctx, cudaSetDevice(d->device));
  const mtb::FlatScene &f = ctx->flat;
  MTB_CUDA(ctx, d->nodes.Upload(f.nodes.data(), f.nodes.size(), d->stream));
  MTB_CUDA(ctx, d->slots.Upload(f.slots.data(), f.slots.size(), d->stream));
  MTB_CUDA(ctx, d->shade.Upload(f.shade.data(), f.shade.size(), d->stream));
  MTB_CUDA(ctx, d->bvh.Upload(f.bvh.data(), f.bvh.size(), d->stream));
  MTB_CUDA(ctx, d->list_order.Upload(f.list_order.data(), f.list_order.size(), d->stream));
  MTB_CUDA(ctx, d->slot_node.Upload(f.slot_node.data(), f.slot_node.size(), d->stream));
  d->gnodes.Free();
  d->gslots.Free();
  d->leaf_ref.Free();
  d->ref_slot.Free();
  d->device_bvh_depth = 0;
  if (ctx->device_bvh) {
    // SURVEY section 8 f1: the scene BVH is built on the device from the reference boxes (PLOC, device_build.cu) and
    // the leaf-ordered triangle records are gathered on the device from the records uploaded above - the host neither
    // builds nor uploads them.
    const auto t0 = std::chrono::steady_clock::now();
    mtb::Bvh2Node *d_nodes = nullptr;
    int32_t *d_leaf_ref = nullptr;
    int32_t n_nodes = 0, depth = 0;
    const int64_t n_refs = (int64_t)f.ref_slot.size();
    const cudaError_t e = mtb::BuildSceneBvhOnDevice(f.ref_box.data(), n_refs, f.aabb, f.bvh_pad, d->stream, &d_nodes, &n_nodes, &d_leaf_ref, &depth);
    if (e != cudaSuccess) {
      cudaGetLastError();
      ctx->err = std::string("device BVH build: ") + cudaGetErrorString(e);
      return MTB_ERR_CUDA;
    }
    d->gnodes.ptr = d_nodes;
    d->gnodes.count = (size_t)n_nodes;
    d->leaf_ref.ptr = d_leaf_ref;
    d->leaf_ref.count = (size_t)n_refs;
    d->device_bvh_depth = depth;
    if (depth > mtb::kSceneBvhMaxDepth) {  // deeper than the traversal stack (never seen): no fast traversal
      d->gnodes.Free();
      d->leaf_ref.Free();
    } else {
      MTB_CUDA(ctx, d->ref_slot.Upload(f.ref_slot.data(), f.ref_slot.size(), d->stream));
      MTB_CUDA(ctx, d->gslots.Reserve((size_t)n_refs));
      mtb::LaunchGatherLeafSlots(d->slots.ptr, d->ref_slot.ptr, d->leaf_ref.ptr, n_refs, d->gslots.ptr, d->stream);
      MTB_CUDA(ctx, cudaGetLastError());
    }
    MTB_CUDA(ctx, cudaStreamSynchronize(d->stream));
    ctx->ms_device_bvh = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (getenv("MTB_TIMING") != nullptr) {
      fprintf(stderr, "[mtb] %-28s %8.1f ms (%d nodes, depth %d)\n", "scene BVH on the device", ctx->ms_device_bvh, n_nodes, depth);
    }
  } else {
    MTB_CUDA(ctx, d->gnodes.Upload(f.gnodes.data(), f.gnodes.size(), d->stream));
    MTB_CUDA(ctx, d->gslots.Upload(f.gslots.data(), f.gslots.size(), d->stream));
    if (f.gnodes.empty()) {
      d->gnodes.Free();
      d->gslots.Free();
    }
  }
  MTB_CUDA(ctx, d->materials.Upload(ctx->materials.data(), ctx->materials.size(), d->stream));
  DestroyTextures(d);
  // All textures live in ONE layered CUDA array behind ONE texture object (layer = texture index, extent = the
  // largest texture; a fetch never leaves its own texture's width x height).  The object is a kernel argument, so
  // the handle is uniform across the warp: per-texture objects fetched from memory made the compiler emit a
  // waterfall loop around every TEX, and that code returned wrong texels in the megakernel.
  std::vector<int2> dims;
  d->scene.tex_atlas = 0;
  if (!ctx->textures.empty()) {
    size_t max_w = 1, max_h = 1;
    for (const mtb::LoadedTexture &t : ctx->textures) {
      max_w = std::max(max_w, (size_t)t.width);
      max_h = std::max(max_h, (size_t)t.height);
      dims.push_back(make_int2(t.width, t.height));
    }
    cudaChannelFormatDesc desc = cudaCreateChannelDesc<unsigned int>();  // one RGBA32 texel = one 32-bit word
    cudaArray_t arr = nullptr;
    // every layer has the extent of the largest texture: what is really allocated is max_w * max_h * layers texels
    // (mtb_scene_info reports that, not the sum of the images), and a scene that mixes one huge texture with many
    // small ones is refused with a clear message instead of a bare CUDA allocation error
    const size_t atlas_bytes = max_w * max_h * ctx->textures.size() * 4;
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && atlas_bytes > free_b) {
      ctx->err = "texture atlas of " + std::to_string(ctx->textures.size()) + " layers of " + std::to_string(max_w) + " x " +
                 std::to_string(max_h) + " texels (" + std::to_string(atlas_bytes >> 20) + " MiB: every layer has the extent of the largest texture) does not fit the device";
      return MTB_ERR_LIMIT;
    }
    ctx->atlas_bytes = (int64_t)atlas_bytes;
    MTB_CUDA(ctx, cudaMalloc3DArray(&arr, &desc, make_cudaExtent(max_w, max_h, ctx->textures.size()), cudaArrayLayered));
    d->tex_arrays.push_back(arr);
    for (size_t layer = 0; layer < ctx->textures.size(); layer++) {
      const mtb::LoadedTexture &t = ctx->textures[layer];
      if (t.width <= 0 || t.height <= 0) continue;
      cudaMemcpy3DParms cp;
      memset(&cp, 0, sizeof(cp));
      cp.srcPtr = make_cudaPitchedPtr(const_cast<uint8_t *>(t.rgba.data()), (size_t)t.width * 4, (size_t)t.width, (size_t)t.height);
      cp.dstArray = arr;
      cp.dstPos = make_cudaPos(0, 0, layer);
      cp.extent = make_cudaExtent((size_t)t.width, (size_t)t.height, 1);
      cp.kind = cudaMemcpyHostToDevice;
      MTB_CUDA(ctx, cudaMemcpy3DAsync(&cp, d->stream));
    }
    cudaResourceDesc res;
    memset(&res, 0, sizeof(res));
    res.resType = cudaResourceTypeArray;
    res.res.array.array = arr;
    cudaTextureDesc td;
    memset(&td, 0, sizeof(td));
    td.addressMode[0] = td.addressMode[1] = td.addressMode[2] = cudaAddressModeClamp;
    td.filterMode = cudaFilterModePoint;  // bilinear weights are done in FP64 by the kernel (texture.cc:47-57)
    td.readMode = cudaReadModeElementType;
    td.normalizedCoords = 0;
    cudaTextureObject_t obj = 0;
    MTB_CUDA(ctx, cudaCreateTextureObject(&obj, &res, &td, nullptr));
    d->tex_handles.push_back(obj);
    d->scene.tex_atlas = obj;
  }
  MTB_CUDA(ctx, d->tex_dims.Upload(dims.data(), dims.size(), d->stream));
  MTB_CUDA(ctx, cudaStreamSynchronize(d->stream));
  d->scene.nodes = d->nodes.ptr;
  d->scene.slots = d->slots.ptr;
  d->scene.shade = d->shade.ptr;
  d->scene.bvh = d->bvh.ptr;
  d->scene.list_order = d->list_order.ptr;
  d->scene.slot_node = d->slot_node.ptr;
  d->scene.materials = d->materials.ptr;
  d->scene.texture_dim = d->tex_dims.ptr;
  d->scene.n_materials = (int32_t)ctx->materials.size();
  d->scene.n_nodes = (int32_t)ctx->flat.nodes.size();
  // the FP32 cull's error bound assumes coordinates of ordinary magnitude (see device_core.cuh, CullBox32 / FastBox)
  const double mac = ctx->flat.max_abs_coord;
  d->scene.cull_radius = (mac >= 0x1p-10 && mac <= 0x1p20) ? (float)mac * 1.0000002f : 0.0f;
  d->scene.max_tri_extent = std::nextafterf((float)ctx->flat.max_tri_extent, INFINITY);
  SelectTraversal(ctx, d);
  return MTB_OK;
}

// A/B knob: an access-policy window over the scene BVH's node array on `s` (hit = persisting, miss = streaming), so
// that the thread-local memory traffic of the kernels cannot evict the nodes every ray walks.
void ApplyL2Window(mtb_context *ctx, DeviceState *d, cudaStream_t s) {
  if (ctx->l2_persist_mb <= 0 || d->gnodes.ptr == nullptr || ctx->flat.gnodes.empty()) return;
  int max_persist = 0, max_window = 0;
  cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, d->device);
  cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, d->device);
  size_t carve = std::min<size_t>((size_t)ctx->l2_persist_mb << 20, (size_t)std::max(max_persist, 0));
  if (carve == 0 || max_window <= 0) return;
  cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve);
  const size_t bytes = std::min<size_t>(ctx->flat.gnodes.size() * sizeof(mtb::Bvh2Node), (size_t)max_window);
  cudaStreamAttrValue attr;
  memset(&attr, 0, sizeof(attr));
  attr.accessPolicyWindow.base_ptr = d->gnodes.ptr;
  attr.accessPolicyWindow.num_bytes = bytes;
  attr.accessPolicyWindow.hitRatio = bytes <= carve ? 1.0f : (float)((double)carve / (double)bytes);
  attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
  attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
  cudaStreamSetAttribute(s, cudaStreamAttributeAccessPolicyWindow, &attr);
  cudaGetLastError();
}

int UploadLights(mtb_context *ctx, DeviceState *d) {
  MTB_CUDA(ctx, cudaSetDevice(d->device));
  MTB_CUDA(ctx, d->lights.Upload(ctx->lights.data(), ctx->lights.size(), d->stream));
  d->scene.lights = d->lights.ptr;
  d->scene.n_lights = (int32_t)ctx->lights.size();
  return MTB_OK;
}

int BuildAndUpload(mtb_context *ctx) {
  // material / texture indices are validated here so the kernels never read out of range
  for (mtb_triangle &t : ctx->triangles) {
    if (t.material < -1 || t.material >= (int32_t)ctx->materials.size()) {
      ctx->err = "triangle references a material outside the table";
      return MTB_ERR_ARG;
    }
  }
  for (mtb_material &m : ctx->materials) {
    if (m.texture < -1 || m.texture >= (int32_t)ctx->textures.size()) {
      ctx->err = "material references a texture outside the table";
      return MTB_ERR_ARG;
    }
  }
  std::string err;
  // Where the scene BVH is built: on the host threads (binned SAH; the default: its trees render C3 12 % faster),
  // on the devices (MTB_FLAG_DEVICE_BVH: PLOC, csrc/device_build.cu; contexts with a device, scenes of at least 64
  // triangles), or not at all (MTB_FLAG_NO_LIST_BVH).
  mtb::SceneBvhMode mode = mtb::kSceneBvhNone;
  if ((ctx->flags & MTB_FLAG_NO_LIST_BVH) == 0) {
    const bool device = !ctx->dev.empty() && (ctx->flags & MTB_FLAG_DEVICE_BVH) != 0 && ctx->triangles.size() >= 64;
    mode = device ? mtb::kSceneBvhRefs : mtb::kSceneBvhHost;
  }
  ctx->device_bvh = mode == mtb::kSceneBvhRefs;
  const int rc = mtb::BuildFlatScene(ctx->triangles.data(), (int64_t)ctx->triangles.size(),
                                     (ctx->flags & MTB_FLAG_NO_LIST_BVH) == 0, mode, &ctx->flat, &err);
  if (rc != MTB_OK) {
    ctx->err = err;
    return rc;
  }
  ctx->device_bytes = (int64_t)(ctx->flat.nodes.size() * sizeof(mtb::NodeRec) + ctx->flat.slots.size() * sizeof(mtb::SlotRec) +
                                ctx->flat.shade.size() * sizeof(mtb::ShadeRec) + ctx->flat.bvh.size() * sizeof(mtb::BvhRec) +
                                ctx->flat.gnodes.size() * sizeof(mtb::Bvh2Node) + ctx->flat.gslots.size() * sizeof(mtb::SlotRec) +
                                ctx->flat.ref_slot.size() * (sizeof(mtb::SlotRec) + 8) +
                                ctx->flat.list_order.size() * 4 + ctx->flat.slot_node.size() * 4 + ctx->materials.size() * sizeof(mtb_material));
  ctx->atlas_bytes = 0;
  const auto t_up = std::chrono::steady_clock::now();
  ctx->ms_device_bvh = 0.0;
  for (DeviceState &d : ctx->dev) {
    const int urc = UploadToDevice(ctx, &d);
    if (urc != MTB_OK) return urc;
  }
  ctx->ms_upload = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_up).count() - ctx->ms_device_bvh;
  if (ctx->device_bvh && !ctx->dev.empty()) ctx->device_bytes += (int64_t)(ctx->dev[0].gnodes.count * sizeof(mtb::Bvh2Node));
  ctx->device_bytes += ctx->atlas_bytes;  // the layered texture array as allocated
  if (getenv("MTB_TIMING") != nullptr) fprintf(stderr, "[mtb] %-28s %8.1f ms\n", "upload", ctx->ms_upload);
  ctx->has_scene = true;
  return MTB_OK;
}

void FillStats(const unsigned long long *c, mtb_stats *s) {
  s->rays = c[mtb::kRays];
  s->primary = c[mtb::kPrimary];
  s->shadow = c[mtb::kShadow];
  s->reflect = c[mtb::kReflect];
  s->refract = c[mtb::kRefract];
  s->n_slab = c[mtb::kSlab];
  s->n_visit = c[mtb::kVisit];
  s->n_triaabb = c[mtb::kTriAabb];
  s->n_mt = c[mtb::kMt];
  s->n_hit = c[mtb::kHit];
  s->n_shade = c[mtb::kShade];
  s->n_bvh = c[mtb::kBvh];
  s->n_literal = c[mtb::kLiteral];
  s->n_fast = c[mtb::kFast];
  s->n_fallback = c[mtb::kFallback];
  s->n_long128_rays = c[mtb::kLongRays128];
  s->n_long128_visits = c[mtb::kLongVisits128];
  s->n_long512_rays = c[mtb::kLongRays512];
  s->n_long512_visits = c[mtb::kLongVisits512];
}

struct StripPlan {
  int n_strips = 0;   // strips of 8 rows in the chunk
  int owners = 1;     // part_count * n_devices
};

// Strips owned by (part p, device g): s % owners == p * n_devices + g.
int OwnedStrips(const StripPlan &plan, int owner) {
  if (owner >= plan.n_strips) return 0;
  return (plan.n_strips - owner + plan.owners - 1) / plan.owners;
}

// Copies the strips that `owner` rendered from its buffer into device 0's buffer (same layout) with one
// pitched peer copy (NVLink when peer access is enabled): rows of the 2-D copy are whole strips.
int GatherStrips(mtb_context *ctx, const StripPlan &plan, int owner, int chunk_w, int chunk_h, size_t elem_bytes,
                 void *dst_base, const void *src_base, cudaStream_t stream) {
  const int mine = OwnedStrips(plan, owner);
  if (mine == 0) return MTB_OK;
  const size_t strip_bytes = (size_t)8 * chunk_w * elem_bytes;
  const size_t pitch = strip_bytes * plan.owners;
  const size_t first = strip_bytes * owner;
  // all owned strips except possibly a clipped last one
  int full = mine;
  const int last_strip = owner + (mine - 1) * plan.owners;
  const int last_rows = chunk_h - last_strip * 8;
  if (last_rows < 8) full = mine - 1;
  if (full > 0) {
    MTB_CUDA(ctx, cudaMemcpy2DAsync(static_cast<char *>(dst_base) + first, pitch,
                                    static_cast<const char *>(src_base) + first, pitch, strip_bytes, (size_t)full,
                                    cudaMemcpyDeviceToDevice, stream));
  }
  if (full < mine) {
    const size_t off = strip_bytes * last_strip;
    MTB_CUDA(ctx, cudaMemcpyAsync(static_cast<char *>(dst_base) + off, static_cast<const char *>(src_base) + off,
                                  (size_t)last_rows * chunk_w * elem_bytes, cudaMemcpyDeviceToDevice, stream));
  }
  return MTB_OK;
}

// Sizes the wavefront buffers for `slots` pixel slots and the current light count.
int EnsureWavefront(mtb_context *ctx, DeviceState *d, int slots, int n_lights) {
  const size_t qcap = (size_t)slots * d->wf_queue_factor;
  const size_t acap = (size_t)slots * d->wf_act_factor;
  if (qcap > 0x7fffffffull / 4 || acap > 0x7fffffffull / 4) {
    ctx->err = "wavefront buffers exceed the 32-bit index range";
    return MTB_ERR_LIMIT;
  }
  for (int k = 0; k < 2; k++) {
    MTB_CUDA(ctx, d->wf_rq_o[k].Reserve(qcap * 3));
    MTB_CUDA(ctx, d->wf_rq_d[k].Reserve(qcap * 3));
    MTB_CUDA(ctx, d->wf_rq_coef[k].Reserve(qcap));
    MTB_CUDA(ctx, d->wf_rq_path[k].Reserve(qcap));
    MTB_CUDA(ctx, d->wf_rq_pixel[k].Reserve(qcap));
    MTB_CUDA(ctx, d->wf_rq_inobj[k].Reserve(qcap));
    d->wf.rq_o[k] = d->wf_rq_o[k].ptr;
    d->wf.rq_d[k] = d->wf_rq_d[k].ptr;
    d->wf.rq_coef[k] = d->wf_rq_coef[k].ptr;
    d->wf.rq_path[k] = d->wf_rq_path[k].ptr;
    d->wf.rq_pixel[k] = d->wf_rq_pixel[k].ptr;
    d->wf.rq_inobj[k] = d->wf_rq_inobj[k].ptr;
  }
  const size_t nl = (size_t)(n_lights > 0 ? n_lights : 1);
  MTB_CUDA(ctx, d->wf_act_point.Reserve(acap * 3));
  MTB_CUDA(ctx, d->wf_act_normal.Reserve(acap * 3));
  MTB_CUDA(ctx, d->wf_act_surface.Reserve(acap * 3));
  MTB_CUDA(ctx, d->wf_act_reflected.Reserve(acap * 3));
  MTB_CUDA(ctx, d->wf_act_dir.Reserve(acap * 3));
  MTB_CUDA(ctx, d->wf_sh_power.Reserve(acap * 3 * nl));
  MTB_CUDA(ctx, d->wf_sh_flags.Reserve(acap * nl));
  MTB_CUDA(ctx, d->wf_act_color.Reserve(acap * 3));
  MTB_CUDA(ctx, d->wf_act_refl.Reserve(acap));
  MTB_CUDA(ctx, d->wf_act_refr.Reserve(acap));
  MTB_CUDA(ctx, d->wf_act_mtl.Reserve(acap));
  MTB_CUDA(ctx, d->wf_act_pixel.Reserve(acap));
  MTB_CUDA(ctx, d->wf_act_path.Reserve(acap));
  if (d->wf_stream2 == nullptr) {
    MTB_CUDA(ctx, cudaStreamCreateWithFlags(&d->wf_stream2, cudaStreamNonBlocking));
    for (cudaStream_t &st : d->wf_side) MTB_CUDA(ctx, cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    for (cudaEvent_t &e : d->wf_ev_side) MTB_CUDA(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (cudaEvent_t &e : d->wf_ev_level) MTB_CUDA(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    MTB_CUDA(ctx, cudaEventCreateWithFlags(&d->wf_ev_lit, cudaEventDisableTiming));
  }
  MTB_CUDA(ctx, d->wf_level_n.Reserve(MTB_MAX_RAY_DEPTH + 2));
  MTB_CUDA(ctx, d->wf_ctrl.Reserve(2));
  MTB_CUDA(ctx, d->wf_work.Reserve(mtb::kNumCounters));
  if (d->wf_host == nullptr) {
    MTB_CUDA(ctx, cudaMallocHost(reinterpret_cast<void **>(&d->wf_host), mtb::kWfHostWords * sizeof(uint32_t)));
    memset(d->wf_host, 0, mtb::kWfHostWords * sizeof(uint32_t));
  }
  d->wf.act_point = d->wf_act_point.ptr;
  d->wf.act_normal = d->wf_act_normal.ptr;
  d->wf.act_surface = d->wf_act_surface.ptr;
  d->wf.act_reflected = d->wf_act_reflected.ptr;
  d->wf.act_dir = d->wf_act_dir.ptr;
  d->wf.sh_power = d->wf_sh_power.ptr;
  d->wf.sh_flags = d->wf_sh_flags.ptr;
  d->wf.act_color = d->wf_act_color.ptr;
  d->wf.act_refl = d->wf_act_refl.ptr;
  d->wf.act_refr = d->wf_act_refr.ptr;
  d->wf.act_mtl = d->wf_act_mtl.ptr;
  d->wf.act_pixel = d->wf_act_pixel.ptr;
  d->wf.act_path = d->wf_act_path.ptr;
  d->wf.level_n = d->wf_level_n.ptr;
  d->wf.ctrl = d->wf_ctrl.ptr;
  d->wf.work = d->wf_work.ptr;
  d->wf.queue_cap = (int32_t)qcap;
  d->wf.act_cap = (int32_t)acap;
  return MTB_OK;
}

// One frame (this device's strips / its share of a hybrid frame) through the wavefront pipeline: every kernel of
// every level is enqueued at once, nothing is read back.  How many rays a level holds is only known on the device;
// the grids are sized from the counts of the last completed frame of the same size (+25 %), else from the capacity
// bound, and the kernels loop grid-strided over the real count.  If a queue overflows, the kernels of the remaining
// levels exit at once and the RenderMega launch queued at the end renders the same tiles instead (same bytes); the
// host sees the overflow flag at the start of the next frame and doubles the queues.
int RunWavefront(mtb_context *ctx, DeviceState *d, const mtb::RenderParams &p, int n_blocks, bool debug_build,
                 cudaStream_t s) {
  const int slots = n_blocks * 64;
  if (slots <= 0) return MTB_OK;
  // feedback of the frames completed so far (pinned memory written by WfCommit; a frame still in flight simply is not
  // in it yet)
  long long hint[MTB_MAX_RAY_DEPTH + 2];
  bool have_hint = false;
  if (d->wf_host != nullptr) {
    const uint32_t seq = d->wf_host[mtb::kWfHostSequence];
    if (seq != d->wf_seen_sequence) {
      d->wf_seen_sequence = seq;
      if (d->wf_host[mtb::kWfHostOverflow] != 0u) {
        d->wf_queue_factor *= 2;
        d->wf_act_factor *= 2;
      }
    }
    if (seq != 0u && d->wf_host[mtb::kWfHostOverflow] == 0u && d->wf_host[0] == (uint32_t)slots) {
      have_hint = true;
      for (int l = 0; l <= MTB_MAX_RAY_DEPTH + 1; l++) hint[l] = (long long)d->wf_host[l];
    }
  }
  const int rc = EnsureWavefront(ctx, d, slots, d->scene.n_lights);
  if (rc != MTB_OK) return rc;
  long long expect[MTB_MAX_RAY_DEPTH + 2];
  for (int level = 0; level <= p.max_depth; level++) {
    long long bound = level >= 24 ? (long long)d->wf.queue_cap : std::min<long long>((long long)d->wf.queue_cap, (long long)slots << level);
    expect[level] = have_hint ? std::min(bound, hint[level] + hint[level] / 4 + 2048) : bound;
  }
  expect[0] = slots;
  // Side streams: the shadow walks + Phong sums of level L only depend on the trace of level L, so the levels'
  // side kernels go round-robin over four streams and overlap each other as well as the deeper traces (on a small
  // share of a frame - one of 8 GPUs - every one of them is latency-bound and they were the critical path when
  // serialised on one stream).
  cudaStream_t side[4] = {d->wf_stream2, d->wf_side[0], d->wf_side[1], d->wf_side[2]};
  mtb::LaunchWfBegin(d->wf, slots, s);
  // they must not start before earlier work on the main stream (previous frame, taps memset, WfBegin)
  MTB_CUDA(ctx, cudaEventRecord(d->wf_ev_lit, s));
  for (cudaStream_t st : side) MTB_CUDA(ctx, cudaStreamWaitEvent(st, d->wf_ev_lit, 0));
  for (int level = 0; level <= p.max_depth; level++) {
    // critical path (main stream): trace the level and queue its children
    mtb::LaunchWfTrace(d->scene, p, d->wf, level, expect[level], debug_build, s);
    MTB_CUDA(ctx, cudaEventRecord(d->wf_ev_level[level], s));
    // side branch: shadow walks and the Phong sums of this level
    cudaStream_t s2 = side[level & 3];
    MTB_CUDA(ctx, cudaStreamWaitEvent(s2, d->wf_ev_level[level], 0));
    mtb::LaunchWfShadow(d->scene, p, d->wf, level, expect[level], debug_build, s2);
    mtb::LaunchWfLight(d->scene, p, d->wf, level, expect[level], s2);
    ctx->launches += 2u + (d->scene.n_lights > 0 ? 1u : 0u);
  }
  // join: the folds need every level's colours
  for (int k = 0; k < 4; k++) {
    MTB_CUDA(ctx, cudaEventRecord(d->wf_ev_side[k], side[k]));
    MTB_CUDA(ctx, cudaStreamWaitEvent(s, d->wf_ev_side[k], 0));
  }
  for (int level = p.max_depth - 1; level >= 0; level--) {
    mtb::LaunchWfFold(d->scene, d->wf, level, expect[level], s);
    ctx->launches++;
  }
  mtb::LaunchWfResolve(p, d->wf, slots, s);
  mtb::LaunchWfCommit(d->wf, p.counters, d->wf_host, s);
  // the repair launch: a no-op (its blocks read one word and exit) unless a queue overflowed
  mtb::RenderParams repair = p;
  repair.run_if = d->wf.ctrl;
  repair.mega_part = 1;
  mtb::LaunchRenderMega(d->scene, repair, n_blocks, debug_build, s);
  ctx->launches += 4u;  // WfBegin, WfResolve, WfCommit, repair
  MTB_CUDA(ctx, cudaGetLastError());
  return MTB_OK;
}

// One frame through the queue pipeline: one persistent kernel takes every activation of every level from a single
// device-side ray queue (wavefront.cu, WfQueue), then the per-pixel fold.  Four launches, nothing read back; overflow
// of the activation table is handled like in RunWavefront (repair launch, larger tables next frame).
int RunWavefrontQueue(mtb_context *ctx, DeviceState *d, const mtb::RenderParams &p, int n_blocks, bool debug_build, cudaStream_t s) {
  const int slots = n_blocks * 64;
  if (slots <= 0) return MTB_OK;
  if (d->wf_host != nullptr) {
    const uint32_t seq = d->wf_host[mtb::kWfHostSequence];
    if (seq != d->wf_seen_sequence) {
      d->wf_seen_sequence = seq;
      if (d->wf_host[mtb::kWfHostOverflow] != 0u) {
        d->wf_queue_factor *= 2;
        d->wf_act_factor *= 2;
      }
    }
  }
  const int rc = EnsureWavefront(ctx, d, slots, d->scene.n_lights);
  if (rc != MTB_OK) return rc;
  const size_t acap = (size_t)d->wf.act_cap;
  const uint32_t *ready_before = d->wf_act_ready.ptr;
  MTB_CUDA(ctx, d->wf_act_coef.Reserve(acap));
  MTB_CUDA(ctx, d->wf_act_info.Reserve(acap));
  MTB_CUDA(ctx, d->wf_act_ready.Reserve(acap));
  MTB_CUDA(ctx, d->wf_qctl.Reserve(mtb::kQWords));
  if (d->wf_act_ready.ptr != ready_before || d->wf_epoch == 0xffffffffu) {
    MTB_CUDA(ctx, cudaMemsetAsync(d->wf_act_ready.ptr, 0, d->wf_act_ready.count * sizeof(uint32_t), s));
    d->wf_epoch = 0;
  }
  d->wf_epoch++;
  d->wf.act_coef = d->wf_act_coef.ptr;
  d->wf.act_info = d->wf_act_info.ptr;
  d->wf.act_ready = d->wf_act_ready.ptr;
  d->wf.qctl = d->wf_qctl.ptr;
  mtb::LaunchWfQueueBegin(d->wf, slots, s);
  mtb::LaunchWfQueue(d->scene, p, d->wf, slots, d->wf_epoch, d->sm_count, debug_build, s);
  mtb::LaunchWfResolveTree(d->scene, p, d->wf, slots, s);
  mtb::LaunchWfCommit(d->wf, p.counters, d->wf_host, s);
  mtb::RenderParams repair = p;
  repair.run_if = d->wf.ctrl;
  repair.mega_part = 1;
  mtb::LaunchRenderMega(d->scene, repair, n_blocks, debug_build, s);
  ctx->launches += 5u;
  MTB_CUDA(ctx, cudaGetLastError());
  return MTB_OK;
}

// Hybrid frames: which tiles go through the wavefront.  The megakernel's critical path is its most expensive pixel
// (a serial chain of up to ~80 rays), the wavefront's is one ray per level but it pays ~1.3x the instructions, so the
// most expensive tiles of the previous frame go to the wavefront and the rest to the megakernel, concurrently.  How
// much is not a constant: round 1 used two fixed rules picked from a table measured on C3; now the share of the
// frame's rays that the wavefront gets is STEERED - both halves are timed with events, and the share moves a step
// towards whichever half finished first (no host wait: the events of the previous frame are only read if they have
// completed).  At most half of the tiles can go to the wavefront (its queues are sized for that).
constexpr int kTuneDecided = 13;  // frames 5..12 of a new geometry are hybrid frames
constexpr float kHybridShareMin = 0.02f, kHybridShareMax = 0.90f, kHybridShareStep = 0.04f;
int HybridMaxTiles(int tiles) { return tiles / 2; }

// Core of both render entry points.  d_rgb_user: device-0 buffer to leave the pixels in (may be NULL when
// rgb_host is given); user_stream: stream of device 0 to enqueue on (NULL = context stream).
int RenderImpl(mtb_context *ctx, const mtb_camera *cam, int image_w, int image_h, int chunk_x, int chunk_y,
               int chunk_w, int chunk_h, int max_depth, uint8_t *rgb_host, void *d_rgb_user, cudaStream_t user_stream,
               mtb_debug *dbg_host, const mtb_taps *taps, mtb_stats *stats, bool synchronous) {
  const auto wall0 = std::chrono::steady_clock::now();
  if (ctx == nullptr) return MTB_ERR_ARG;
  if (ctx->dev.empty()) {
    ctx->err = "host-only context: no CUDA device to render on (there is no CPU fallback)";
    return MTB_ERR_CUDA;
  }
  if (!ctx->has_scene) {
    ctx->err = "no scene uploaded";
    return MTB_ERR_ARG;
  }
  if (cam == nullptr || image_w <= 0 || image_h <= 0 || chunk_w <= 0 || chunk_h <= 0 || chunk_x < 0 || chunk_y < 0 ||
      max_depth < 0 || max_depth > MTB_MAX_RAY_DEPTH) {
    ctx->err = "bad render arguments";
    return MTB_ERR_ARG;
  }
  const size_t npx = (size_t)chunk_w * chunk_h;
  const bool want_taps = taps != nullptr && (taps->sig_hits || taps->sig_shadow || taps->n_rays);
  const bool debug_build = (ctx->flags & MTB_FLAG_COUNT_WORK) != 0;
  const int n_dev = (int)ctx->dev.size();
  StripPlan plan;
  plan.n_strips = (chunk_h + 7) / 8;
  plan.owners = ctx->part_count * n_dev;

  mtb::RenderParams rp;
  memset(&rp, 0, sizeof(rp));
  mtb::ComputeSensor(*cam, image_w, image_h, rp.sensor);
  for (int a = 0; a < 3; a++) rp.origin[a] = cam->origin[a];
  rp.image_w = image_w;
  rp.image_h = image_h;
  rp.chunk_x = chunk_x;
  rp.chunk_y = chunk_y;
  rp.chunk_w = chunk_w;
  rp.chunk_h = chunk_h;
  rp.max_depth = max_depth;
  rp.tiles_x = (chunk_w + 7) / 8;
  rp.strip_stride = plan.owners;

  // the frame on device 0 that receives every device's tiles
  DeviceState &dev0 = ctx->dev[0];
  MTB_CUDA(ctx, cudaSetDevice(dev0.device));
  // A pinned host frame (mtb_host_alloc, cudaHostAlloc, a registered buffer) is mapped into the device's address space
  // under unified addressing: with one device the kernels then store their finished tile rows (aligned 8-byte stores)
  // straight into it over PCIe, overlapped with the rendering, and the frame-sized device-to-host copy at the end of
  // the step disappears.  Pageable host memory and multi-device contexts take the copy.  MTB_NO_HOST_STORE=1 is the A/B.
  uint8_t *host_direct = nullptr;
  if (rgb_host != nullptr && d_rgb_user == nullptr && n_dev == 1 && !ctx->no_host_store && (chunk_w & 7) == 0 &&
      (reinterpret_cast<uintptr_t>(rgb_host) & 7u) == 0u) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, rgb_host) == cudaSuccess && attr.type == cudaMemoryTypeHost && attr.devicePointer != nullptr) {
      host_direct = static_cast<uint8_t *>(attr.devicePointer);
    }
    cudaGetLastError();  // (an unregistered pointer is not an error here)
  }
  if (d_rgb_user == nullptr && host_direct == nullptr) MTB_CUDA(ctx, dev0.rgb.Reserve(npx * 3));
  uint8_t *const rgb_target = d_rgb_user != nullptr ? static_cast<uint8_t *>(d_rgb_user) : (host_direct != nullptr ? host_direct : dev0.rgb.ptr);
  // direct peer stores need a mapping of the target in the storing device's address space: the context's own frame
  // (cudaMalloc) has one wherever peer access is on; a caller's buffer may come from an allocator without one
  std::vector<char> peer_store((size_t)n_dev, 0);
  for (int g = 1; g < n_dev; g++) peer_store[(size_t)g] = ctx->dev[(size_t)g].peer_store_dev0 && d_rgb_user == nullptr && !ctx->no_peer_store;

  // ---- launch on every device: one host thread per device when there are several (launching a frame is a few
  // dozen driver calls per device; in parallel the devices start together) ----
  auto launch_on_device = [&](int g) -> int {
    DeviceState &d = ctx->dev[g];
    MTB_CUDA(ctx, cudaSetDevice(d.device));
    cudaStream_t s = (g == 0 && user_stream != nullptr) ? user_stream : d.stream;
    const int owner = ctx->part_index * n_dev + g;
    mtb::RenderParams p = rp;
    p.strip_first = owner;
    // Where the pixels go.  Device 0: the caller's device buffer, or the context's frame.  Other devices: straight
    // into device 0's frame through its peer mapping when there is one (RenderMega leaves whole tile rows as aligned
    // 8-byte stores, WfResolve likewise) - the in-box BlitWorkChunk (main_net_master.cc:223-236) costs no copy then -
    // else into an own frame that device 0 gathers with one pitched peer copy.
    if (g == 0) {
      p.rgb = rgb_target;
    } else if (peer_store[(size_t)g]) {
      p.rgb = rgb_target;
    } else {
      MTB_CUDA(ctx, d.rgb.Reserve(npx * 3));
      p.rgb = d.rgb.ptr;
    }
    if (dbg_host != nullptr) {
      MTB_CUDA(ctx, d.dbg.Reserve(npx));
      p.dbg = d.dbg.ptr;
    }
    if (want_taps) {
      MTB_CUDA(ctx, d.sig_hits.Reserve(npx));
      MTB_CUDA(ctx, d.sig_shadow.Reserve(npx));
      MTB_CUDA(ctx, d.n_rays.Reserve(npx));
      p.sig_hits = d.sig_hits.ptr;
      p.sig_shadow = d.sig_shadow.ptr;
      p.n_rays = d.n_rays.ptr;
    }
    MTB_CUDA(ctx, d.counters.Reserve(mtb::kNumCounters));
    p.counters = d.counters.ptr;
    if (stats != nullptr || synchronous) {
      MTB_CUDA(ctx, cudaMemsetAsync(d.counters.ptr, 0, mtb::kNumCounters * sizeof(unsigned long long), s));
    }
    const int blocks = OwnedStrips(plan, owner) * rp.tiles_x;
    // a peer's scratch frame must not be overwritten while device 0 still gathers the previous one
    if (g > 0) MTB_CUDA(ctx, cudaStreamWaitEvent(s, ctx->dev[0].ev_gathered, 0));
    bool wavefront = (ctx->flags & (MTB_FLAG_WAVEFRONT | MTB_FLAG_QUEUE)) != 0;
    bool queue = (ctx->flags & MTB_FLAG_QUEUE) != 0;  // the wavefront as one persistent kernel over a ray queue
    bool hybrid = (ctx->flags & MTB_FLAG_HYBRID) != 0 && !wavefront;
    if ((ctx->flags & (MTB_FLAG_WAVEFRONT | MTB_FLAG_QUEUE | MTB_FLAG_MEGAKERNEL | MTB_FLAG_HYBRID)) == 0 && blocks > 0) {
      // automatic: measure both pipelines on the first frames of this geometry, then keep the faster
      const long long tsig = ((long long)chunk_w << 42) ^ ((long long)chunk_h << 24) ^ ((long long)owner << 12) ^
                             ((long long)plan.owners << 6) ^ ((long long)max_depth << 1) ^ ((long long)d.scene.n_lights << 50);
      if (tsig != d.tune_signature) {
        d.tune_signature = tsig;
        d.tune_stage = 0;
      } else if (d.tune_stage == 2 || d.tune_stage == 4 || d.tune_stage == kTuneDecided - 1) {
        // the previous frame was a timed one: harvest it
        float ms = 0.f;
        if (cudaEventSynchronize(d.ev_stop) == cudaSuccess && cudaEventElapsedTime(&ms, d.ev_start, d.ev_stop) == cudaSuccess) {
          d.tune_ms[d.tune_stage == 2 ? 0 : (d.tune_stage == 4 ? 1 : 2)] = ms;
        }
        if (d.tune_stage == kTuneDecided - 1) {
          d.tune_choice = 0;
          if (d.tune_ms[1] < d.tune_ms[d.tune_choice]) d.tune_choice = 1;
          if (d.tune_ms[2] < d.tune_ms[d.tune_choice]) d.tune_choice = 2;
        }
      }
      if (d.tune_stage < kTuneDecided) d.tune_stage++;
      // stage now: 1 = megakernel (cold tile order), 2 = megakernel (timed), 3 = queue pipeline (cold: buffers are
      // allocated), 4 = queue pipeline (timed), 5 .. kTuneDecided - 1 = hybrid (the split settles; the last one is
      // timed), kTuneDecided = decided.  (The wavefront candidate is its queue form: measured faster than the
      // level-by-level form at every share of the C3 frame, DESIGN.md section 6.)
      wavefront = d.tune_stage == 3 || d.tune_stage == 4 || (d.tune_stage == kTuneDecided && d.tune_choice == 1);
      queue = wavefront;
      hybrid = (d.tune_stage >= 5 && d.tune_stage < kTuneDecided) || (d.tune_stage == kTuneDecided && d.tune_choice == 2);
    }
    if (ctx->l2_persist_mb > 0 && d.l2_window_stream != s) {
      ApplyL2Window(ctx, &d, s);
      d.l2_window_stream = s;
    }
    MTB_CUDA(ctx, cudaEventRecord(d.ev_start, s));
    if (wavefront) {
      // the wavefront kernels accumulate the taps with atomics
      if (want_taps) {
        MTB_CUDA(ctx, cudaMemsetAsync(d.sig_hits.ptr, 0, npx * 8, s));
        MTB_CUDA(ctx, cudaMemsetAsync(d.sig_shadow.ptr, 0, npx * 8, s));
        MTB_CUDA(ctx, cudaMemsetAsync(d.n_rays.ptr, 0, npx * 4, s));
      }
      const int wrc = queue ? RunWavefrontQueue(ctx, &d, p, blocks, debug_build, s) : RunWavefront(ctx, &d, p, blocks, debug_build, s);
      if (wrc != MTB_OK) return wrc;
    } else {
      const int mblocks = blocks;
      if (mblocks > 0 && (ctx->flags & MTB_FLAG_NO_TILE_ORDER) == 0) {
        // launch order from the previous frame of the same geometry; the first frame runs in scanline order
        const long long signature = ((long long)chunk_w << 40) ^ ((long long)chunk_h << 20) ^ ((long long)owner << 8) ^ plan.owners ^
                                    ((long long)mblocks << 4);
        MTB_CUDA(ctx, d.tile_cost.Reserve((size_t)mblocks));
        MTB_CUDA(ctx, d.tile_order.Reserve((size_t)mblocks));
        p.tile_cost = d.tile_cost.ptr;
        const bool split = hybrid && mblocks >= 64;
        if (split) MTB_CUDA(ctx, d.heavy_k.Reserve(1));
        if (split && d.hybrid_timed && d.ev_wf_done != nullptr && cudaEventQuery(d.ev_wf_done) == cudaSuccess &&
            cudaEventQuery(d.ev_mega_done) == cudaSuccess) {
          // steer the split with the previous hybrid frame: the half that took longer gives up work
          float t_mega = 0.f, t_wf = 0.f;
          if (cudaEventElapsedTime(&t_mega, d.ev_split, d.ev_mega_done) == cudaSuccess &&
              cudaEventElapsedTime(&t_wf, d.ev_split, d.ev_wf_done) == cudaSuccess) {
            if (t_wf > t_mega * 1.04f) d.hybrid_share -= kHybridShareStep;
            if (t_mega > t_wf * 1.04f) d.hybrid_share += kHybridShareStep;
            d.hybrid_share = std::min(kHybridShareMax, std::max(kHybridShareMin, d.hybrid_share));
          }
          cudaGetLastError();
        }
        if (signature == d.tile_signature) {
          mtb::LaunchBuildTileOrder(d.tile_cost.ptr, d.tile_order.ptr, mblocks, split ? d.heavy_k.ptr : nullptr, HybridMaxTiles(mblocks),
                                    (unsigned)(d.hybrid_share * 65536.0f), s);
          ctx->launches++;
          p.tile_order = d.tile_order.ptr;
          if (split) p.heavy_k = d.heavy_k.ptr;
        } else {
          MTB_CUDA(ctx, cudaMemsetAsync(d.tile_cost.ptr, 0, (size_t)mblocks * sizeof(uint32_t), s));
          d.tile_signature = signature;
          d.hybrid_timed = false;
        }
      }
      if (p.heavy_k != nullptr) {
        // Hybrid frame.  The megakernel's critical path is its most expensive pixel (a serial chain of up to ~80
        // rays), the wavefront's is one ray per level but it pays ~1.3x the instructions: so the tiles that were
        // the most expensive in the previous frame (the first *heavy_k of the launch order, at most 1/8 of the tiles)
        // go through the wavefront while the megakernel renders the rest on a second stream.  Both write their own
        // pixels of the same buffers; the bytes do not depend on the split.
        if (d.hybrid_stream == nullptr) {
          MTB_CUDA(ctx, cudaStreamCreateWithFlags(&d.hybrid_stream, cudaStreamNonBlocking));
          MTB_CUDA(ctx, cudaEventCreate(&d.ev_split));
          MTB_CUDA(ctx, cudaEventCreate(&d.ev_mega_done));
          MTB_CUDA(ctx, cudaEventCreate(&d.ev_wf_done));
        }
        if (want_taps) {  // the wavefront kernels accumulate the taps with atomics
          MTB_CUDA(ctx, cudaMemsetAsync(d.sig_hits.ptr, 0, npx * 8, s));
          MTB_CUDA(ctx, cudaMemsetAsync(d.sig_shadow.ptr, 0, npx * 8, s));
          MTB_CUDA(ctx, cudaMemsetAsync(d.n_rays.ptr, 0, npx * 4, s));
        }
        MTB_CUDA(ctx, cudaEventRecord(d.ev_split, s));
        MTB_CUDA(ctx, cudaStreamWaitEvent(d.hybrid_stream, d.ev_split, 0));
        mtb::LaunchRenderMega(d.scene, p, mblocks, debug_build, d.hybrid_stream);
        ctx->launches++;
        MTB_CUDA(ctx, cudaGetLastError());
        MTB_CUDA(ctx, cudaEventRecord(d.ev_mega_done, d.hybrid_stream));
        const int wrc = RunWavefront(ctx, &d, p, HybridMaxTiles(mblocks), debug_build, s);
        if (wrc != MTB_OK) return wrc;
        MTB_CUDA(ctx, cudaEventRecord(d.ev_wf_done, s));
        d.hybrid_timed = true;
        MTB_CUDA(ctx, cudaStreamWaitEvent(s, d.ev_mega_done, 0));
      } else {
        mtb::LaunchRenderMega(d.scene, p, mblocks, debug_build, s);
        if (mblocks > 0) ctx->launches++;
        MTB_CUDA(ctx, cudaGetLastError());
      }
    }
    MTB_CUDA(ctx, cudaEventRecord(d.ev_stop, s));
    return MTB_OK;
  };
  if (n_dev == 1) {
    const int rc = launch_on_device(0);
    if (rc != MTB_OK) return rc;
  } else {
    std::vector<int> rcs((size_t)n_dev, MTB_OK);
    std::vector<std::thread> workers;
    for (int g = 0; g < n_dev; g++) workers.emplace_back([&, g]() { rcs[(size_t)g] = launch_on_device(g); });
    for (std::thread &t : workers) t.join();
    for (int rc : rcs) {
      if (rc != MTB_OK) return rc;
    }
  }

  // ---- gather on device 0 (peer copies), then device -> host ----
  DeviceState &d0 = ctx->dev[0];
  MTB_CUDA(ctx, cudaSetDevice(d0.device));
  cudaStream_t s0 = user_stream != nullptr ? user_stream : d0.stream;
  uint8_t *rgb0 = rgb_target;
  for (int g = 1; g < n_dev; g++) {
    DeviceState &d = ctx->dev[g];
    const int owner = ctx->part_index * n_dev + g;
    MTB_CUDA(ctx, cudaStreamWaitEvent(s0, d.ev_stop, 0));
    int rc = peer_store[(size_t)g] ? MTB_OK : GatherStrips(ctx, plan, owner, chunk_w, chunk_h, 3, rgb0, d.rgb.ptr, s0);
    if (rc != MTB_OK) return rc;
    if (dbg_host != nullptr) {
      rc = GatherStrips(ctx, plan, owner, chunk_w, chunk_h, sizeof(mtb_debug), d0.dbg.ptr, d.dbg.ptr, s0);
      if (rc != MTB_OK) return rc;
    }
    if (want_taps) {
      rc = GatherStrips(ctx, plan, owner, chunk_w, chunk_h, 8, d0.sig_hits.ptr, d.sig_hits.ptr, s0);
      if (rc == MTB_OK) rc = GatherStrips(ctx, plan, owner, chunk_w, chunk_h, 8, d0.sig_shadow.ptr, d.sig_shadow.ptr, s0);
      if (rc == MTB_OK) rc = GatherStrips(ctx, plan, owner, chunk_w, chunk_h, 4, d0.n_rays.ptr, d.n_rays.ptr, s0);
      if (rc != MTB_OK) return rc;
    }
  }
  if (rgb_host != nullptr && host_direct == nullptr) MTB_CUDA(ctx, cudaMemcpyAsync(rgb_host, rgb0, npx * 3, cudaMemcpyDeviceToHost, s0));
  if (dbg_host != nullptr) {
    MTB_CUDA(ctx, cudaMemcpyAsync(dbg_host, d0.dbg.ptr, npx * sizeof(mtb_debug), cudaMemcpyDeviceToHost, s0));
  }
  if (want_taps) {
    if (taps->sig_hits) MTB_CUDA(ctx, cudaMemcpyAsync(taps->sig_hits, d0.sig_hits.ptr, npx * 8, cudaMemcpyDeviceToHost, s0));
    if (taps->sig_shadow) MTB_CUDA(ctx, cudaMemcpyAsync(taps->sig_shadow, d0.sig_shadow.ptr, npx * 8, cudaMemcpyDeviceToHost, s0));
    if (taps->n_rays) MTB_CUDA(ctx, cudaMemcpyAsync(taps->n_rays, d0.n_rays.ptr, npx * 4, cudaMemcpyDeviceToHost, s0));
  }
  // the peers may overwrite their scratch frames, and device 0's frame, once this frame has left device 0
  if (n_dev > 1) MTB_CUDA(ctx, cudaEventRecord(d0.ev_gathered, s0));
  if (!synchronous && stats == nullptr) return MTB_OK;

  MTB_CUDA(ctx, cudaStreamSynchronize(s0));
  if (stats != nullptr) {
    unsigned long long total[mtb::kNumCounters];
    memset(total, 0, sizeof(total));
    double kernel_ms = 0.0;
    for (int g = 0; g < n_dev; g++) {
      DeviceState &d = ctx->dev[g];
      MTB_CUDA(ctx, cudaSetDevice(d.device));
      cudaStream_t s = (g == 0 && user_stream != nullptr) ? user_stream : d.stream;
      MTB_CUDA(ctx, cudaStreamSynchronize(s));
      unsigned long long c[mtb::kNumCounters];
      MTB_CUDA(ctx, cudaMemcpy(c, d.counters.ptr, sizeof(c), cudaMemcpyDeviceToHost));
      for (int i = 0; i < mtb::kNumCounters; i++) total[i] += c[i];
      float ms = 0.f;
      MTB_CUDA(ctx, cudaEventElapsedTime(&ms, d.ev_start, d.ev_stop));
      if (ms > kernel_ms) kernel_ms = ms;  // devices run concurrently: the frame takes the slowest
    }
    memset(stats, 0, sizeof(*stats));
    FillStats(total, stats);
    stats->kernel_ms = kernel_ms;
    stats->total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - wall0).count();
  }
  return MTB_OK;
}

// A batch: n_views whole frames of one scene, one camera and one light set per view.  Always the megakernel, in one
// launch per device (grid = tiles of a view x views of the device): the pipeline choice, the cost-aware tile order, the
// hybrid split and the strip interleave are all single-frame machinery and none of their state is read or written.
// lights == NULL: every view uses the context's lights.  Device g renders a contiguous range of views; the counts
// differ by at most one.  ss > 1 (samples per axis, 2, 4 or 8): every view is traced on the (ss*W) x (ss*H) sample grid,
// exactly as a batch of that size, and the kernel writes the W x H block means; everything else is as for ss = 1.
constexpr int64_t kMaxSampleSide = 65536;  // (keeps the tiles of a view's sample grid, 2^26, well inside int32)
int RenderBatchImpl(mtb_context *ctx, const mtb_camera *cams, int32_t n_views, const mtb_light *lights, int32_t n_lights, int image_w,
                    int image_h, int ss, int max_depth, uint8_t *rgb_host, mtb_stats *stats, bool synchronous) {
  const auto wall0 = std::chrono::steady_clock::now();
  if (ctx == nullptr) return MTB_ERR_ARG;
  if (ctx->dev.empty()) {
    ctx->err = "host-only context: no CUDA device to render on (there is no CPU fallback)";
    return MTB_ERR_CUDA;
  }
  if (!ctx->has_scene) {
    ctx->err = "no scene uploaded";
    return MTB_ERR_ARG;
  }
  if (cams == nullptr || rgb_host == nullptr) {
    ctx->err = cams == nullptr ? "cams is NULL" : "rgb_out is NULL";
    return MTB_ERR_ARG;
  }
  if (n_views < 1 || n_views > 65535) {
    ctx->err = "n_views must be in 1..65535 (one grid row per view)";
    return MTB_ERR_ARG;
  }
  if (lights != nullptr && n_lights < 0) {
    ctx->err = "n_lights must be >= 0";
    return MTB_ERR_ARG;
  }
  if (image_w <= 0 || image_h <= 0 || max_depth < 0 || max_depth > MTB_MAX_RAY_DEPTH) {
    ctx->err = "bad render arguments";
    return MTB_ERR_ARG;
  }
  if (ss != 1 && ss != 2 && ss != 4 && ss != 8) {
    ctx->err = "samples_per_axis must be 1, 2, 4 or 8 (the samples of an output pixel then lie in one 8x8 tile)";
    return MTB_ERR_ARG;
  }
  if (ss > 1 && ((int64_t)image_w * ss > kMaxSampleSide || (int64_t)image_h * ss > kMaxSampleSide)) {
    ctx->err = "the sample grid (samples_per_axis * image_w x samples_per_axis * image_h) must be at most 65536 on a side";
    return MTB_ERR_ARG;
  }
  if (ctx->part_index != 0 || ctx->part_count != 1) {
    ctx->err = "a batch renders whole views: the partition must be (0, 1)";
    return MTB_ERR_ARG;
  }
  const size_t npx = (size_t)image_w * image_h;  // output pixels of a view
  const int grid_w = image_w * ss, grid_h = image_h * ss;  // its sample grid (the view itself when ss = 1)
  const bool debug_build = (ctx->flags & MTB_FLAG_COUNT_WORK) != 0;
  const int n_dev = (int)ctx->dev.size();
  const int tiles_x = (grid_w + 7) / 8, tiles_per_view = tiles_x * ((grid_h + 7) / 8);

  // per-view records and the views' lights, view-major (the context's lights repeated when the caller passes none)
  const int32_t nl = lights != nullptr ? n_lights : (int32_t)ctx->lights.size();
  std::vector<mtb::ViewRec> views((size_t)n_views);
  std::vector<mtb_light> view_lights((size_t)n_views * nl);
  for (int32_t v = 0; v < n_views; v++) {
    mtb::ComputeSensor(cams[v], grid_w, grid_h, views[(size_t)v].sensor);
    for (int a = 0; a < 3; a++) views[(size_t)v].origin[a] = cams[v].origin[a];
    const mtb_light *src = lights != nullptr ? lights + (size_t)v * nl : ctx->lights.data();
    if (nl > 0) std::copy(src, src + nl, view_lights.begin() + (size_t)v * nl);
  }

  mtb::RenderParams rp;
  memset(&rp, 0, sizeof(rp));
  rp.image_w = rp.chunk_w = grid_w;
  rp.image_h = rp.chunk_h = grid_h;
  rp.max_depth = max_depth;
  rp.tiles_x = tiles_x;
  rp.strip_stride = 1;

  // Where the pixels go: a single device stores straight into a mapped pinned rgb_host (RenderImpl's rule); otherwise
  // every device renders into its own frames and copies its views to their slice of rgb_host.  Supersampled views always
  // take the second way: their epilogue stores single bytes, and a direct store of those into mapped host memory has
  // not been measured against the copy (which moves 1/ss^2 of the samples' bytes).
  uint8_t *host_direct = nullptr;
  if (ss == 1 && n_dev == 1 && !ctx->no_host_store && (image_w & 7) == 0 && (reinterpret_cast<uintptr_t>(rgb_host) & 7u) == 0u) {
    MTB_CUDA(ctx, cudaSetDevice(ctx->dev[0].device));
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, rgb_host) == cudaSuccess && attr.type == cudaMemoryTypeHost && attr.devicePointer != nullptr) {
      host_direct = static_cast<uint8_t *>(attr.devicePointer);
    }
    cudaGetLastError();  // (an unregistered pointer is not an error here)
  }

  auto launch_on_device = [&](int g) -> int {
    DeviceState &d = ctx->dev[(size_t)g];
    const int first = g * (n_views / n_dev) + std::min(g, n_views % n_dev);
    const int count = n_views / n_dev + (g < n_views % n_dev ? 1 : 0);
    if (count == 0) return MTB_OK;
    MTB_CUDA(ctx, cudaSetDevice(d.device));
    cudaStream_t s = d.stream;
    if (d.ev_batch_start == nullptr) {
      MTB_CUDA(ctx, cudaEventCreate(&d.ev_batch_start));
      MTB_CUDA(ctx, cudaEventCreate(&d.ev_batch_stop));
    }
    // Everything below is ordered on d.stream: a batch queued behind another one overwrites the records only after the
    // earlier launch has read them.  A buffer that has to grow is freed and reallocated, so the earlier work that may
    // still read it is waited for first.
    const size_t n_rgb = host_direct != nullptr ? 0 : (size_t)count * npx * 3;
    const size_t n_lt = (size_t)count * nl;
    if ((size_t)count > d.batch_views.count || n_lt > d.batch_lights.count || n_rgb > d.batch_rgb.count) {
      MTB_CUDA(ctx, cudaStreamSynchronize(s));
    }
    MTB_CUDA(ctx, d.batch_views.Upload(views.data() + first, (size_t)count, s));
    MTB_CUDA(ctx, d.batch_lights.Upload(view_lights.data() + (size_t)first * nl, n_lt, s));
    if (n_rgb > 0) MTB_CUDA(ctx, d.batch_rgb.Reserve(n_rgb));
    mtb::DeviceScene sc = d.scene;
    sc.lights = d.batch_lights.ptr;
    sc.n_lights = nl;
    mtb::RenderParams p = rp;
    p.rgb = host_direct != nullptr ? host_direct + (size_t)first * npx * 3 : d.batch_rgb.ptr;
    MTB_CUDA(ctx, d.counters.Reserve(mtb::kNumCounters));
    p.counters = d.counters.ptr;
    if (stats != nullptr || synchronous) {
      MTB_CUDA(ctx, cudaMemsetAsync(d.counters.ptr, 0, mtb::kNumCounters * sizeof(unsigned long long), s));
    }
    MTB_CUDA(ctx, cudaEventRecord(d.ev_batch_start, s));
    mtb::LaunchRenderMegaBatch(sc, p, d.batch_views.ptr, tiles_per_view, count, ss, debug_build, s);
    ctx->launches++;
    MTB_CUDA(ctx, cudaGetLastError());
    MTB_CUDA(ctx, cudaEventRecord(d.ev_batch_stop, s));
    if (host_direct == nullptr) {
      MTB_CUDA(ctx, cudaMemcpyAsync(rgb_host + (size_t)first * npx * 3, d.batch_rgb.ptr, (size_t)count * npx * 3, cudaMemcpyDeviceToHost, s));
    }
    return MTB_OK;
  };
  if (n_dev == 1) {
    const int rc = launch_on_device(0);
    if (rc != MTB_OK) return rc;
  } else {
    std::vector<int> rcs((size_t)n_dev, MTB_OK);
    std::vector<std::thread> workers;
    for (int g = 0; g < n_dev; g++) workers.emplace_back([&, g]() { rcs[(size_t)g] = launch_on_device(g); });
    for (std::thread &t : workers) t.join();
    for (int rc : rcs) {
      if (rc != MTB_OK) return rc;
    }
  }
  if (!synchronous && stats == nullptr) return MTB_OK;

  unsigned long long total[mtb::kNumCounters];
  memset(total, 0, sizeof(total));
  double kernel_ms = 0.0;
  for (int g = 0; g < n_dev && g < n_views; g++) {
    DeviceState &d = ctx->dev[(size_t)g];
    MTB_CUDA(ctx, cudaSetDevice(d.device));
    MTB_CUDA(ctx, cudaStreamSynchronize(d.stream));
    if (stats == nullptr) continue;
    unsigned long long c[mtb::kNumCounters];
    MTB_CUDA(ctx, cudaMemcpy(c, d.counters.ptr, sizeof(c), cudaMemcpyDeviceToHost));
    for (int i = 0; i < mtb::kNumCounters; i++) total[i] += c[i];
    float ms = 0.f;
    MTB_CUDA(ctx, cudaEventElapsedTime(&ms, d.ev_batch_start, d.ev_batch_stop));
    if (ms > kernel_ms) kernel_ms = ms;  // devices run concurrently: the batch takes the slowest
  }
  if (stats != nullptr) {
    memset(stats, 0, sizeof(*stats));
    FillStats(total, stats);
    stats->kernel_ms = kernel_ms;
    stats->total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - wall0).count();
  }
  return MTB_OK;
}

}  // namespace

extern "C" {

const char *mtb_version(void) { return "mythtracer_b200 0.1 (sm_100a)"; }

int mtb_create(mtb_context **out, const int *devices, int n_devices) {
  if (out == nullptr) return MTB_ERR_ARG;
  *out = nullptr;
  int available = 0;
  cudaError_t e = cudaGetDeviceCount(&available);
  if (e != cudaSuccess || available == 0) {
    g_create_error = std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "count is 0");
    return MTB_ERR_CUDA;
  }
  mtb_context *ctx = new mtb_context;
  const int n = (devices == nullptr || n_devices <= 0) ? 1 : n_devices;
  ctx->dev.resize((size_t)n);
  for (int g = 0; g < n; g++) {
    DeviceState &d = ctx->dev[(size_t)g];
    d.device = (devices == nullptr || n_devices <= 0) ? 0 : devices[g];
    if (d.device < 0 || d.device >= available) {
      g_create_error = "device ordinal out of range";
      delete ctx;
      return MTB_ERR_ARG;
    }
    if ((e = cudaSetDevice(d.device)) != cudaSuccess || (e = cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking)) != cudaSuccess ||
        (e = cudaEventCreate(&d.ev_start)) != cudaSuccess || (e = cudaEventCreate(&d.ev_stop)) != cudaSuccess ||
        (e = cudaEventCreateWithFlags(&d.ev_gathered, cudaEventDisableTiming)) != cudaSuccess) {
      g_create_error = std::string("device setup failed: ") + cudaGetErrorString(e);
      delete ctx;
      return MTB_ERR_CUDA;
    }
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, d.device) == cudaSuccess && sms > 0) d.sm_count = sms;
  }
  // NVLink peer access between device 0, the gather target, and every other device: device 0 -> g for the peer-copy
  // gather of taps / debug planes, g -> device 0 so that g's kernels can store their tiles straight into the frame
  for (int g = 1; g < n; g++) {
    int can = 0;
    cudaDeviceCanAccessPeer(&can, ctx->dev[0].device, ctx->dev[(size_t)g].device);
    if (can) {
      cudaSetDevice(ctx->dev[0].device);
      e = cudaDeviceEnablePeerAccess(ctx->dev[(size_t)g].device, 0);
      if (e == cudaSuccess || e == cudaErrorPeerAccessAlreadyEnabled) ctx->dev[(size_t)g].peer_to_dev0 = true;
      cudaGetLastError();
    }
    can = 0;
    cudaDeviceCanAccessPeer(&can, ctx->dev[(size_t)g].device, ctx->dev[0].device);
    if (can) {
      cudaSetDevice(ctx->dev[(size_t)g].device);
      e = cudaDeviceEnablePeerAccess(ctx->dev[0].device, 0);
      if (e == cudaSuccess || e == cudaErrorPeerAccessAlreadyEnabled) ctx->dev[(size_t)g].peer_store_dev0 = true;
      cudaGetLastError();
    }
  }
  {  // development knobs (A/B measurements, tests that force a queue overflow)
    const char *v = getenv("MTB_NO_PEER_STORE");
    ctx->no_peer_store = v != nullptr && v[0] == '1';
    const char *hs = getenv("MTB_NO_HOST_STORE");
    ctx->no_host_store = hs != nullptr && hs[0] == '1';
    const char *l2 = getenv("MTB_L2_PERSIST_MB");
    ctx->l2_persist_mb = l2 != nullptr ? atoi(l2) : 0;
    const char *qf = getenv("MTB_WF_QUEUE_FACTOR"), *af = getenv("MTB_WF_ACT_FACTOR");
    for (DeviceState &d : ctx->dev) {
      if (qf != nullptr && atoi(qf) >= 1) d.wf_queue_factor = atoi(qf);
      if (af != nullptr && atoi(af) >= 1) d.wf_act_factor = atoi(af);
    }
  }
  *out = ctx;
  return MTB_OK;
}

int mtb_create_host(mtb_context **out) {
  if (out == nullptr) return MTB_ERR_ARG;
  *out = new mtb_context;
  return MTB_OK;
}

void mtb_destroy(mtb_context *ctx) {
  if (ctx == nullptr) return;
  if (!ctx->dev.empty()) {
    cudaSetDevice(ctx->dev[0].device);
    cudaDeviceSynchronize();
    for (void *p : ctx->opened_frames) cudaIpcCloseMemHandle(p);
    for (void *p : ctx->owned_frames) cudaFree(p);
  }
  for (DeviceState &d : ctx->dev) {
    cudaSetDevice(d.device);
    if (d.stream != nullptr) cudaStreamSynchronize(d.stream);
    DestroyTextures(&d);
    d.FreeAll();
    if (d.ev_start != nullptr) cudaEventDestroy(d.ev_start);
    if (d.ev_stop != nullptr) cudaEventDestroy(d.ev_stop);
    if (d.ev_gathered != nullptr) cudaEventDestroy(d.ev_gathered);
    if (d.stream != nullptr) cudaStreamDestroy(d.stream);
  }
  delete ctx;
}

const char *mtb_last_error(const mtb_context *ctx) { return ctx == nullptr ? g_create_error.c_str() : ctx->err.c_str(); }

int mtb_device_count(const mtb_context *ctx) { return ctx == nullptr ? 0 : (int)ctx->dev.size(); }

int mtb_scene_upload(mtb_context *ctx, const mtb_triangle *tris, int64_t n_tris, const mtb_material *mtls,
                     int32_t n_mtls, const mtb_texture *texs, int32_t n_texs) {
  if (ctx == nullptr || n_tris < 0 || n_mtls < 0 || n_texs < 0 || (n_tris > 0 && tris == nullptr) ||
      (n_mtls > 0 && mtls == nullptr) || (n_texs > 0 && texs == nullptr)) {
    if (ctx != nullptr) ctx->err = "bad scene arguments";
    return MTB_ERR_ARG;
  }
  ctx->has_scene = false;
  ctx->triangles.assign(tris, tris + n_tris);
  ctx->materials.assign(mtls, mtls + n_mtls);
  ctx->textures.clear();
  ctx->material_names.clear();
  ctx->texture_names.clear();
  for (int32_t i = 0; i < n_texs; i++) {
    if (texs[i].width <= 0 || texs[i].height <= 0 || texs[i].rgba == nullptr) {
      ctx->err = "bad texture";
      return MTB_ERR_ARG;
    }
    mtb::LoadedTexture t;
    t.width = texs[i].width;
    t.height = texs[i].height;
    t.rgba.assign(texs[i].rgba, texs[i].rgba + (size_t)t.width * t.height * 4);
    ctx->textures.push_back(std::move(t));
  }
  return BuildAndUpload(ctx);
}

int mtb_load_obj(mtb_context *ctx, const char *path) {
  if (ctx == nullptr || path == nullptr) return MTB_ERR_ARG;
  mtb::LoadedScene loaded;
  std::string err;
  ctx->has_scene = false;
  const auto t_parse = std::chrono::steady_clock::now();
  const bool parsed = mtb::LoadObjFile(path, &loaded, &err);
  ctx->ms_parse = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_parse).count();
  if (getenv("MTB_TIMING") != nullptr) fprintf(stderr, "[mtb] %-28s %8.1f ms\n", "OBJ + MTL parse", ctx->ms_parse);
  if (!parsed) {
    ctx->err = err;
    fprintf(stderr, "error: %s\n", err.c_str());
    return MTB_ERR_IO;
  }
  ctx->triangles.swap(loaded.triangles);
  ctx->materials.swap(loaded.materials);
  ctx->textures.swap(loaded.textures);
  ctx->material_names.swap(loaded.material_names);
  ctx->texture_names.swap(loaded.texture_names);
  return BuildAndUpload(ctx);
}

int mtb_load_mtl(mtb_context *ctx, const char *path) {
  if (ctx == nullptr || path == nullptr) return MTB_ERR_ARG;
  mtb::LoadedScene loaded;
  std::string err;
  ctx->has_scene = false;
  if (!mtb::LoadMtlFile(path, &loaded, &err)) {
    ctx->err = err;
    fprintf(stderr, "error: %s\n", err.c_str());
    return MTB_ERR_IO;
  }
  ctx->triangles.clear();
  ctx->materials.swap(loaded.materials);
  ctx->textures.swap(loaded.textures);
  ctx->material_names.swap(loaded.material_names);
  ctx->texture_names.swap(loaded.texture_names);
  return BuildAndUpload(ctx);
}

const char *mtb_scene_material_name(const mtb_context *ctx, int32_t index) {
  if (ctx == nullptr || index < 0 || (size_t)index >= ctx->material_names.size()) return nullptr;
  return ctx->material_names[(size_t)index].c_str();
}

const char *mtb_scene_texture_name(const mtb_context *ctx, int32_t index) {
  if (ctx == nullptr || index < 0 || (size_t)index >= ctx->texture_names.size()) return nullptr;
  return ctx->texture_names[(size_t)index].c_str();
}

int mtb_scene_texture(const mtb_context *ctx, int32_t index, mtb_texture *out) {
  if (ctx == nullptr || out == nullptr || index < 0 || (size_t)index >= ctx->textures.size()) return MTB_ERR_ARG;
  out->width = ctx->textures[(size_t)index].width;
  out->height = ctx->textures[(size_t)index].height;
  out->rgba = ctx->textures[(size_t)index].rgba.data();
  return MTB_OK;
}

int mtb_set_lights(mtb_context *ctx, const mtb_light *lights, int32_t n) {
  if (ctx == nullptr || n < 0 || (n > 0 && lights == nullptr)) return MTB_ERR_ARG;
  ctx->lights.assign(lights, lights + n);
  for (DeviceState &d : ctx->dev) {
    const int rc = UploadLights(ctx, &d);
    if (rc != MTB_OK) return rc;
    // the render may be enqueued on a caller stream: make the new lights visible first
    MTB_CUDA(ctx, cudaStreamSynchronize(d.stream));
  }
  return MTB_OK;
}

int mtb_scene_info(const mtb_context *ctx, mtb_scene_summary *out) {
  if (ctx == nullptr || out == nullptr) return MTB_ERR_ARG;
  memset(out, 0, sizeof(*out));
  out->n_triangles = (int64_t)ctx->triangles.size();
  out->n_nodes = (int64_t)ctx->flat.nodes.size();
  out->n_bvh_nodes = (int64_t)ctx->flat.bvh.size();
  out->tree_depth = ctx->flat.depth;
  out->n_materials = (int32_t)ctx->materials.size();
  out->n_textures = (int32_t)ctx->textures.size();
  out->n_lights = (int32_t)ctx->lights.size();
  out->root_list = ctx->flat.root_list;
  out->biggest_list = ctx->flat.biggest_list;
  out->interior_triangles = ctx->flat.interior;
  for (int a = 0; a < 3; a++) {
    out->aabb_min[a] = ctx->flat.aabb[a];
    out->aabb_max[a] = ctx->flat.aabb[3 + a];
  }
  out->device_bytes = ctx->device_bytes;
  out->n_scene_refs = ctx->device_bvh ? (int64_t)ctx->flat.ref_slot.size() : (int64_t)ctx->flat.gslots.size();
  return MTB_OK;
}

int mtb_scene_read(const mtb_context *ctx, mtb_triangle *tris, mtb_material *mtls) {
  if (ctx == nullptr) return MTB_ERR_ARG;
  if (tris != nullptr && !ctx->triangles.empty()) memcpy(tris, ctx->triangles.data(), ctx->triangles.size() * sizeof(mtb_triangle));
  if (mtls != nullptr && !ctx->materials.empty()) memcpy(mtls, ctx->materials.data(), ctx->materials.size() * sizeof(mtb_material));
  return MTB_OK;
}

int mtb_scene_triangle_nodes(const mtb_context *ctx, double *node_box, int32_t *node_depth) {
  if (ctx == nullptr) return MTB_ERR_ARG;
  const mtb::FlatScene &f = ctx->flat;
  std::vector<int32_t> depth(f.nodes.size(), 0);
  for (size_t i = 0; i < f.nodes.size(); i++) {
    const mtb::NodeRec &n = f.nodes[i];
    if (n.first_child >= 0) {
      for (int k = 0; k < 8; k++) depth[(size_t)n.first_child + k] = depth[i] + 1;
    }
    for (int32_t k = 0; k < n.list_count; k++) {
      const int32_t tri = f.slots[(size_t)(n.list_first + k)].tri;
      if (node_depth != nullptr) node_depth[tri] = depth[i];
      if (node_box != nullptr) {
        for (int a = 0; a < 3; a++) {
          node_box[(size_t)tri * 6 + a] = n.planes[a];
          node_box[(size_t)tri * 6 + 3 + a] = n.planes[6 + a];
        }
      }
    }
  }
  return MTB_OK;
}

int mtb_scene_bvh(const mtb_context *ctx, int64_t *n_nodes, int32_t *depth, void *nodes, int32_t *leaf_order) {
  if (ctx == nullptr) return MTB_ERR_ARG;
  const mtb::FlatScene &f = ctx->flat;
  if (ctx->device_bvh && !ctx->dev.empty()) {
    // built on the device: read it back from device 0 for inspection
    const DeviceState &d = ctx->dev[0];
    if (n_nodes != nullptr) *n_nodes = (int64_t)d.gnodes.count;
    if (depth != nullptr) *depth = d.device_bvh_depth;
    if (cudaSetDevice(d.device) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) return MTB_ERR_CUDA;
    if (nodes != nullptr && d.gnodes.count > 0 &&
        cudaMemcpy(nodes, d.gnodes.ptr, d.gnodes.count * sizeof(mtb::Bvh2Node), cudaMemcpyDeviceToHost) != cudaSuccess) return MTB_ERR_CUDA;
    if (leaf_order != nullptr && d.leaf_ref.count > 0) {
      std::vector<int32_t> refs(d.leaf_ref.count);
      if (cudaMemcpy(refs.data(), d.leaf_ref.ptr, refs.size() * sizeof(int32_t), cudaMemcpyDeviceToHost) != cudaSuccess) return MTB_ERR_CUDA;
      for (size_t i = 0; i < refs.size(); i++) leaf_order[i] = f.slots[(size_t)f.ref_slot[(size_t)refs[i]]].tri;
    }
    return MTB_OK;
  }
  if (n_nodes != nullptr) *n_nodes = (int64_t)f.gnodes.size();
  if (depth != nullptr) *depth = f.gbvh_depth;
  if (nodes != nullptr && !f.gnodes.empty()) memcpy(nodes, f.gnodes.data(), f.gnodes.size() * sizeof(mtb::Bvh2Node));
  if (leaf_order != nullptr) {
    for (size_t i = 0; i < f.gslots.size(); i++) leaf_order[i] = f.gslots[i].tri;
  }
  return MTB_OK;
}

int mtb_load_timing(const mtb_context *ctx, double out_ms[8]) {
  if (ctx == nullptr || out_ms == nullptr) return MTB_ERR_ARG;
  out_ms[0] = ctx->ms_parse;
  out_ms[1] = ctx->flat.ms_octree;
  out_ms[2] = ctx->flat.ms_flatten;
  out_ms[3] = ctx->flat.ms_scene_bvh;
  out_ms[4] = ctx->ms_device_bvh;
  out_ms[5] = ctx->ms_upload;
  out_ms[6] = ctx->device_bvh ? 1.0 : 0.0;
  out_ms[7] = ctx->flat.ms_scene_bvh_thread;
  return MTB_OK;
}

int mtb_set_flags(mtb_context *ctx, uint32_t flags) {
  if (ctx == nullptr) return MTB_ERR_ARG;
  const bool rebuild = ((ctx->flags ^ flags) & (MTB_FLAG_NO_LIST_BVH | MTB_FLAG_DEVICE_BVH)) != 0 && ctx->has_scene;
  ctx->flags = flags;
  if (rebuild) return BuildAndUpload(ctx);
  for (DeviceState &d : ctx->dev) SelectTraversal(ctx, &d);
  return MTB_OK;
}

int mtb_set_partition(mtb_context *ctx, int part_index, int part_count) {
  if (ctx == nullptr || part_count < 1 || part_index < 0 || part_index >= part_count) return MTB_ERR_ARG;
  ctx->part_index = part_index;
  ctx->part_count = part_count;
  return MTB_OK;
}

int mtb_render_chunk(mtb_context *ctx, const mtb_camera *cam, int image_w, int image_h, int chunk_x, int chunk_y,
                     int chunk_w, int chunk_h, int max_depth, uint8_t *rgb_out, mtb_debug *dbg_out,
                     const mtb_taps *taps, mtb_stats *stats) {
  if (ctx != nullptr && rgb_out == nullptr) {
    ctx->err = "rgb_out is NULL";
    return MTB_ERR_ARG;
  }
  return RenderImpl(ctx, cam, image_w, image_h, chunk_x, chunk_y, chunk_w, chunk_h, max_depth, rgb_out, nullptr, nullptr,
                    dbg_out, taps, stats, true);
}

int mtb_render_chunk_async(mtb_context *ctx, const mtb_camera *cam, int image_w, int image_h, int chunk_x, int chunk_y,
                           int chunk_w, int chunk_h, int max_depth, uint8_t *rgb_out) {
  if (ctx != nullptr && rgb_out == nullptr) {
    ctx->err = "rgb_out is NULL";
    return MTB_ERR_ARG;
  }
  return RenderImpl(ctx, cam, image_w, image_h, chunk_x, chunk_y, chunk_w, chunk_h, max_depth, rgb_out, nullptr, nullptr,
                    nullptr, nullptr, nullptr, false);
}

int mtb_render_batch(mtb_context *ctx, const mtb_camera *cams, int32_t n_views, const mtb_light *lights, int32_t n_lights, int image_w,
                     int image_h, int max_depth, uint8_t *rgb_out, mtb_stats *stats) {
  return RenderBatchImpl(ctx, cams, n_views, lights, n_lights, image_w, image_h, 1, max_depth, rgb_out, stats, true);
}

int mtb_render_batch_async(mtb_context *ctx, const mtb_camera *cams, int32_t n_views, const mtb_light *lights, int32_t n_lights,
                           int image_w, int image_h, int max_depth, uint8_t *rgb_out) {
  return RenderBatchImpl(ctx, cams, n_views, lights, n_lights, image_w, image_h, 1, max_depth, rgb_out, nullptr, false);
}

int mtb_render_batch_ss(mtb_context *ctx, const mtb_camera *cams, int32_t n_views, const mtb_light *lights, int32_t n_lights, int image_w,
                        int image_h, int samples_per_axis, int max_depth, uint8_t *rgb_out, mtb_stats *stats) {
  return RenderBatchImpl(ctx, cams, n_views, lights, n_lights, image_w, image_h, samples_per_axis, max_depth, rgb_out, stats, true);
}

int mtb_render_batch_ss_async(mtb_context *ctx, const mtb_camera *cams, int32_t n_views, const mtb_light *lights, int32_t n_lights,
                              int image_w, int image_h, int samples_per_axis, int max_depth, uint8_t *rgb_out) {
  return RenderBatchImpl(ctx, cams, n_views, lights, n_lights, image_w, image_h, samples_per_axis, max_depth, rgb_out, nullptr, false);
}

int mtb_wait(mtb_context *ctx) {
  if (ctx == nullptr) return MTB_ERR_ARG;
  for (DeviceState &d : ctx->dev) {
    MTB_CUDA(ctx, cudaSetDevice(d.device));
    MTB_CUDA(ctx, cudaStreamSynchronize(d.stream));
  }
  return MTB_OK;
}

void *mtb_host_alloc(size_t bytes) {
  void *p = nullptr;
  if (cudaMallocHost(&p, bytes == 0 ? 1 : bytes) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return p;
}

void mtb_host_free(void *p) {
  if (p != nullptr) cudaFreeHost(p);
}

int mtb_render_chunk_device(mtb_context *ctx, const mtb_camera *cam, int image_w, int image_h, int chunk_x,
                            int chunk_y, int chunk_w, int chunk_h, int max_depth, void *d_rgb, void *stream,
                            mtb_stats *stats) {
  if (ctx != nullptr && d_rgb == nullptr) {
    ctx->err = "d_rgb is NULL";
    return MTB_ERR_ARG;
  }
  return RenderImpl(ctx, cam, image_w, image_h, chunk_x, chunk_y, chunk_w, chunk_h, max_depth, nullptr, d_rgb,
                    static_cast<cudaStream_t>(stream), nullptr, nullptr, stats, false);
}

uint64_t mtb_launch_count(const mtb_context *ctx) { return ctx == nullptr ? 0 : ctx->launches.load(); }

int mtb_pipeline_in_use(const mtb_context *ctx, float *mega_ms, float *wavefront_ms) {
  if (ctx == nullptr || ctx->dev.empty()) return -1;
  const DeviceState &d = ctx->dev[0];
  if (mega_ms != nullptr) *mega_ms = d.tune_ms[0];
  if (wavefront_ms != nullptr) *wavefront_ms = d.tune_ms[1];
  if ((ctx->flags & MTB_FLAG_QUEUE) != 0) return 3;
  if ((ctx->flags & MTB_FLAG_WAVEFRONT) != 0) return 1;
  if ((ctx->flags & MTB_FLAG_HYBRID) != 0) return 2;
  if ((ctx->flags & MTB_FLAG_MEGAKERNEL) != 0) return 0;
  if (d.tune_stage < kTuneDecided) return -1;
  return d.tune_choice == 1 ? 3 : d.tune_choice;
}

float mtb_hybrid_share(const mtb_context *ctx) { return ctx == nullptr || ctx->dev.empty() ? 0.0f : ctx->dev[0].hybrid_share; }

int mtb_read_counters(mtb_context *ctx, mtb_stats *stats) {
  if (ctx == nullptr || stats == nullptr) return MTB_ERR_ARG;
  unsigned long long total[mtb::kNumCounters];
  memset(total, 0, sizeof(total));
  for (DeviceState &d : ctx->dev) {
    MTB_CUDA(ctx, cudaSetDevice(d.device));
    MTB_CUDA(ctx, cudaDeviceSynchronize());
    if (d.counters.ptr == nullptr) continue;
    unsigned long long c[mtb::kNumCounters];
    MTB_CUDA(ctx, cudaMemcpy(c, d.counters.ptr, sizeof(c), cudaMemcpyDeviceToHost));
    MTB_CUDA(ctx, cudaMemset(d.counters.ptr, 0, sizeof(c)));
    for (int i = 0; i < mtb::kNumCounters; i++) total[i] += c[i];
  }
  memset(stats, 0, sizeof(*stats));
  FillStats(total, stats);
  return MTB_OK;
}

int mtb_intersect_rays(mtb_context *ctx, int64_t n, const double *origins, const double *dirs, int32_t *tri_index,
                       double *t, double *point, mtb_stats *stats) {
  const auto wall0 = std::chrono::steady_clock::now();
  if (ctx == nullptr) return MTB_ERR_ARG;
  if (ctx->dev.empty()) {
    ctx->err = "host-only context: no CUDA device to intersect on (there is no CPU fallback)";
    return MTB_ERR_CUDA;
  }
  if (!ctx->has_scene) {
    ctx->err = "no scene uploaded";
    return MTB_ERR_ARG;
  }
  if (n < 0 || (n > 0 && (origins == nullptr || dirs == nullptr || tri_index == nullptr))) {
    ctx->err = "bad intersect arguments";
    return MTB_ERR_ARG;
  }
  if (stats != nullptr) memset(stats, 0, sizeof(*stats));
  if (n == 0) return MTB_OK;
  DeviceState &d = ctx->dev[0];
  MTB_CUDA(ctx, cudaSetDevice(d.device));
  const size_t sn = (size_t)n;
  MTB_CUDA(ctx, d.q_origins.Upload(origins, sn * 3, d.stream));
  MTB_CUDA(ctx, d.q_dirs.Upload(dirs, sn * 3, d.stream));
  MTB_CUDA(ctx, d.q_tri.Reserve(sn));
  MTB_CUDA(ctx, d.q_t.Reserve(sn));
  MTB_CUDA(ctx, d.q_point.Reserve(sn * 3));
  MTB_CUDA(ctx, d.counters.Reserve(mtb::kNumCounters));
  MTB_CUDA(ctx, cudaMemsetAsync(d.counters.ptr, 0, mtb::kNumCounters * sizeof(unsigned long long), d.stream));
  mtb::IntersectParams ip;
  ip.n = n;
  ip.origins = d.q_origins.ptr;
  ip.dirs = d.q_dirs.ptr;
  ip.tri_index = d.q_tri.ptr;
  ip.t = d.q_t.ptr;
  ip.point = d.q_point.ptr;
  ip.counters = d.counters.ptr;
  MTB_CUDA(ctx, cudaEventRecord(d.ev_start, d.stream));
  mtb::LaunchIntersect(d.scene, ip, (ctx->flags & MTB_FLAG_COUNT_WORK) != 0,
                       ((ctx->flags & MTB_FLAG_PAIR_RAYS) != 0 ? 1 : 0) + ((ctx->flags & MTB_FLAG_CHAIN_RAYS) != 0 ? 2 : 0), d.stream);
  ctx->launches++;
  MTB_CUDA(ctx, cudaGetLastError());
  MTB_CUDA(ctx, cudaEventRecord(d.ev_stop, d.stream));
  MTB_CUDA(ctx, cudaMemcpyAsync(tri_index, d.q_tri.ptr, sn * 4, cudaMemcpyDeviceToHost, d.stream));
  if (t != nullptr) MTB_CUDA(ctx, cudaMemcpyAsync(t, d.q_t.ptr, sn * 8, cudaMemcpyDeviceToHost, d.stream));
  if (point != nullptr) MTB_CUDA(ctx, cudaMemcpyAsync(point, d.q_point.ptr, sn * 24, cudaMemcpyDeviceToHost, d.stream));
  MTB_CUDA(ctx, cudaStreamSynchronize(d.stream));
  if (stats != nullptr) {
    unsigned long long c[mtb::kNumCounters];
    MTB_CUDA(ctx, cudaMemcpy(c, d.counters.ptr, sizeof(c), cudaMemcpyDeviceToHost));
    FillStats(c, stats);
    if (stats->rays == 0) stats->rays = (uint64_t)n;
    float ms = 0.f;
    MTB_CUDA(ctx, cudaEventElapsedTime(&ms, d.ev_start, d.ev_stop));
    stats->kernel_ms = ms;
    stats->total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - wall0).count();
  }
  return MTB_OK;
}

// ---- frames shared between processes (one process per GPU) ----
int mtb_frame_create(mtb_context *ctx, size_t bytes, void **d_ptr, unsigned char handle[MTB_FRAME_HANDLE_BYTES]) {
  if (ctx == nullptr || d_ptr == nullptr || handle == nullptr || ctx->dev.empty()) return MTB_ERR_ARG;
  static_assert(sizeof(cudaIpcMemHandle_t) <= MTB_FRAME_HANDLE_BYTES, "handle size");
  *d_ptr = nullptr;
  MTB_CUDA(ctx, cudaSetDevice(ctx->dev[0].device));
  void *p = nullptr;
  MTB_CUDA(ctx, cudaMalloc(&p, bytes == 0 ? 1 : bytes));
  cudaIpcMemHandle_t h;
  const cudaError_t e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) {
    cudaFree(p);
    ctx->err = std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e);
    return MTB_ERR_CUDA;
  }
  MTB_CUDA(ctx, cudaMemset(p, 0, bytes == 0 ? 1 : bytes));
  memset(handle, 0, MTB_FRAME_HANDLE_BYTES);
  memcpy(handle, &h, sizeof(h));
  ctx->owned_frames.push_back(p);
  *d_ptr = p;
  return MTB_OK;
}

int mtb_frame_open(mtb_context *ctx, const unsigned char handle[MTB_FRAME_HANDLE_BYTES], void **d_ptr) {
  if (ctx == nullptr || d_ptr == nullptr || handle == nullptr || ctx->dev.empty()) return MTB_ERR_ARG;
  *d_ptr = nullptr;
  MTB_CUDA(ctx, cudaSetDevice(ctx->dev[0].device));
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  void *p = nullptr;
  MTB_CUDA(ctx, cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
  ctx->opened_frames.push_back(p);
  *d_ptr = p;
  return MTB_OK;
}

int mtb_frame_release(mtb_context *ctx, void *d_ptr) {
  if (ctx == nullptr || d_ptr == nullptr || ctx->dev.empty()) return MTB_ERR_ARG;
  MTB_CUDA(ctx, cudaSetDevice(ctx->dev[0].device));
  for (size_t i = 0; i < ctx->owned_frames.size(); i++) {
    if (ctx->owned_frames[i] == d_ptr) {
      ctx->owned_frames.erase(ctx->owned_frames.begin() + (long)i);
      MTB_CUDA(ctx, cudaFree(d_ptr));
      return MTB_OK;
    }
  }
  for (size_t i = 0; i < ctx->opened_frames.size(); i++) {
    if (ctx->opened_frames[i] == d_ptr) {
      ctx->opened_frames.erase(ctx->opened_frames.begin() + (long)i);
      MTB_CUDA(ctx, cudaIpcCloseMemHandle(d_ptr));
      return MTB_OK;
    }
  }
  ctx->err = "not a frame of this context";
  return MTB_ERR_ARG;
}

int mtb_frame_read(mtb_context *ctx, const void *d_ptr, size_t offset, size_t bytes, void *host_out) {
  if (ctx == nullptr || d_ptr == nullptr || host_out == nullptr || ctx->dev.empty()) return MTB_ERR_ARG;
  MTB_CUDA(ctx, cudaSetDevice(ctx->dev[0].device));
  MTB_CUDA(ctx, cudaDeviceSynchronize());
  MTB_CUDA(ctx, cudaMemcpy(host_out, static_cast<const char *>(d_ptr) + offset, bytes, cudaMemcpyDeviceToHost));
  return MTB_OK;
}

int mtb_camera_sensor(const mtb_camera *cam, int image_w, int image_h, double out9[9]) {
  if (cam == nullptr || out9 == nullptr || image_w <= 0 || image_h <= 0) return MTB_ERR_ARG;
  mtb::ComputeSensor(*cam, image_w, image_h, out9);
  return MTB_OK;
}

}  // extern "C"
