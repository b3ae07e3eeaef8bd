// reference VerStarting/mythtracer.h:8-82 -- the drop-in boundary of the ray-casting path.
//
//   #include <mythtracer/mythtracer.h>      // -I <repo>/include,  link -L<repo>/mythtracer_b200 -lmythtracer_b200
//
// Same names and signatures as the reference (MythTracer::GetScene / LoadObj / RayTrace x2, WorkChunk and its
// four (de)serialisers, PerPixelDebugInfo, MAX_RECURSION_LEVEL); the rendering itself is mtb_render_chunk,
// i.e. hand-written CUDA kernels.  Without a CUDA device RayTrace returns false -- there is no CPU fallback.
#pragma once
#include <stdint.h>

#include <cstdio>
#include <cstring>
#include <limits>
#include <vector>

#include "../mythtracer_b200.h"
#include "camera.h"
#include "objreader.h"
#include "octtree.h"

namespace raytracer {
using math3d::V3D;

const int MAX_RECURSION_LEVEL = 5;  // default; MythTracer::SetMaxRecursionLevel overrides it at run time

struct PerPixelDebugInfo {
  int line_no;
  V3D point;
};
static_assert(sizeof(PerPixelDebugInfo) == sizeof(mtb_debug), "PerPixelDebugInfo layout");
static_assert(sizeof(Light) == sizeof(mtb_light), "Light layout");

class WorkChunk {
 public:
  int image_width, image_height;
  int chunk_x, chunk_y;
  int chunk_width, chunk_height;
  Camera camera;

  static const size_t kSerializedInputSize = 6 * sizeof(uint32_t);
  static const size_t kSerializedOutputMinimumSize = sizeof(uint32_t);

  std::vector<uint8_t> output_bitmap;
  std::vector<PerPixelDebugInfo> output_debug;

  void SerializeInput(std::vector<uint8_t> *bytes) {  // mythtracer.cc:314-333
    const uint32_t f[6] = {(uint32_t)image_width, (uint32_t)image_height, (uint32_t)chunk_x,
                           (uint32_t)chunk_y,     (uint32_t)chunk_width,  (uint32_t)chunk_height};
    bytes->resize(kSerializedInputSize);
    memcpy(bytes->data(), f, sizeof(f));
  }
  bool DeserializeInput(const std::vector<uint8_t> &bytes) {  // mythtracer.cc:335-381
    if (bytes.size() != kSerializedInputSize) return false;
    uint32_t f[6];
    memcpy(f, bytes.data(), sizeof(f));
    const uint32_t iw = f[0], ih = f[1], cx = f[2], cy = f[3], cw = f[4], ch = f[5];
    if (iw > 100000 || ih > 100000 || cx > iw || cy > ih || cw > iw || ch > ih || cx + cw > iw || cy + ch > ih || iw == 0 ||
        ih == 0 || cw == 0 || ch == 0) {
      return false;
    }
    image_width = (int)iw;
    image_height = (int)ih;
    chunk_x = (int)cx;
    chunk_y = (int)cy;
    chunk_width = (int)cw;
    chunk_height = (int)ch;
    return true;
  }
  bool SerializeOutput(std::vector<uint8_t> *bytes) {  // mythtracer.cc:383-397
    if (output_bitmap.size() > std::numeric_limits<uint32_t>::max()) {
      fprintf(stderr, "error: too large WorkerChunk, cannot serialize\n");
      return false;
    }
    const uint32_t sz = (uint32_t)output_bitmap.size();
    bytes->resize(sizeof(uint32_t) + sz);
    memcpy(bytes->data(), &sz, sizeof(sz));
    if (sz > 0) memcpy(bytes->data() + sizeof(sz), output_bitmap.data(), sz);
    return true;
  }
  bool DeserializeOutput(const std::vector<uint8_t> &bytes) {  // mythtracer.cc:399-429
    if (bytes.size() < kSerializedOutputMinimumSize) return false;
    uint32_t sz;
    memcpy(&sz, bytes.data(), sizeof(sz));
    const uint64_t pixels = (uint64_t)chunk_width * (uint64_t)chunk_height;
    if (sz / 3 != pixels || sz % 3 != 0 || bytes.size() - sizeof(sz) < sz) return false;
    output_bitmap.assign(bytes.begin() + sizeof(sz), bytes.begin() + sizeof(sz) + sz);
    return true;
  }
};

class MythTracer {
 public:
  Scene *GetScene() { return &scene; }

  bool LoadObj(const char *fname) {  // mythtracer.cc:247-256
    puts("Reading .OBJ file.");
    ObjFileReader objreader;
    if (!objreader.ReadObjFile(&scene, fname)) return false;
    was_scene_finalized = false;
    return true;
  }

  bool RayTrace(int image_width, int image_height, Camera *camera, std::vector<uint8_t> *output_bitmap) {  // :258-277
    WorkChunk chunk{image_width, image_height, 0, 0, image_width, image_height, *camera, {}, {}};
    chunk.output_bitmap.resize((size_t)image_width * image_height * 3);
    if (!RayTrace(&chunk)) return false;
    *output_bitmap = std::move(chunk.output_bitmap);
    return true;
  }

  // mythtracer.cc:280-312.  chunk->output_bitmap must be pre-sized by the caller (chunk_w * chunk_h * 3), as
  // upstream; a non-empty output_debug (chunk_w * chunk_h entries) receives the primary-hit taps.
  bool RayTrace(WorkChunk *chunk) {
    if (!was_scene_finalized) {
      puts("Finalizing tree.");
      if (!scene.tree.Finalize(&scene.materials, &scene.textures)) return false;
      was_scene_finalized = true;
    }
    puts("Rendering.");
    mtb_context *ctx = scene.tree.context();
    if (chunk->output_bitmap.size() < (size_t)chunk->chunk_width * chunk->chunk_height * 3) return false;
    if (mtb_set_lights(ctx, reinterpret_cast<const mtb_light *>(scene.lights.data()), (int32_t)scene.lights.size()) != MTB_OK) {
      return false;
    }
    const mtb_camera cam = chunk->camera.AsMtb();
    mtb_stats stats;
    const int rc = mtb_render_chunk(
        ctx, &cam, chunk->image_width, chunk->image_height, chunk->chunk_x, chunk->chunk_y, chunk->chunk_width,
        chunk->chunk_height, max_recursion_level, chunk->output_bitmap.data(),
        chunk->output_debug.empty() ? nullptr : reinterpret_cast<mtb_debug *>(chunk->output_debug.data()), nullptr, &stats);
    if (rc != MTB_OK) {
      fprintf(stderr, "error: %s\n", mtb_last_error(ctx));
      return false;
    }
    last_stats = stats;
    printf("%.3fs\n", stats.total_ms * 1e-3);
    return true;
  }

  // ---- extensions ----
  // Frame sequencing: enqueue a whole-frame render into `pinned_out` (w * h * 3 bytes from AllocFrame) and return
  // without waiting; Wait() blocks until it is there.  With two frames in rotation the caller writes frame k while
  // frame k+1 renders (apps/mythtracer_local_b200.cc).
  bool RayTraceAsync(int image_width, int image_height, Camera *camera, uint8_t *pinned_out) {
    if (!was_scene_finalized) {
      puts("Finalizing tree.");
      if (!scene.tree.Finalize(&scene.materials, &scene.textures)) return false;
      was_scene_finalized = true;
    }
    mtb_context *ctx = scene.tree.context();
    if (mtb_set_lights(ctx, reinterpret_cast<const mtb_light *>(scene.lights.data()), (int32_t)scene.lights.size()) != MTB_OK) {
      return false;
    }
    const mtb_camera cam = camera->AsMtb();
    const int rc = mtb_render_chunk_async(ctx, &cam, image_width, image_height, 0, 0, image_width, image_height,
                                          max_recursion_level, pinned_out);
    if (rc != MTB_OK) fprintf(stderr, "error: %s\n", mtb_last_error(ctx));
    return rc == MTB_OK;
  }
  // Batches (mtb_render_batch): cams.size() whole frames in one launch per device, written view-major to `out`
  // (cams.size() * w * h * 3 bytes).  lights: one light list per view, all of the same length; nullptr = scene.lights
  // for every view.  RayTraceBatchAsync returns once the batch is queued (`out` pinned, from AllocFrames; Wait joins).
  bool RayTraceBatch(int image_width, int image_height, const std::vector<Camera> &cams, const std::vector<std::vector<Light>> *lights,
                     uint8_t *out) {
    return RenderBatch(image_width, image_height, 1, cams, lights, out, true);
  }
  bool RayTraceBatchAsync(int image_width, int image_height, const std::vector<Camera> &cams, const std::vector<std::vector<Light>> *lights,
                          uint8_t *pinned_out) {
    return RenderBatch(image_width, image_height, 1, cams, lights, pinned_out, false);
  }
  // Anti-aliased batches (mtb_render_batch_ss): samples_per_axis s = 1, 2, 4 or 8; every output pixel is the rounded
  // mean of the s x s pixels of the same view rendered at (s*w) x (s*h).  `out` holds cams.size() * w * h * 3 bytes.
  bool RayTraceBatch(int image_width, int image_height, int samples_per_axis, const std::vector<Camera> &cams,
                     const std::vector<std::vector<Light>> *lights, uint8_t *out) {
    return RenderBatch(image_width, image_height, samples_per_axis, cams, lights, out, true);
  }
  bool RayTraceBatchAsync(int image_width, int image_height, int samples_per_axis, const std::vector<Camera> &cams,
                          const std::vector<std::vector<Light>> *lights, uint8_t *pinned_out) {
    return RenderBatch(image_width, image_height, samples_per_axis, cams, lights, pinned_out, false);
  }
  bool Wait() { return mtb_wait(scene.tree.context()) == MTB_OK; }
  static uint8_t *AllocFrames(int image_width, int image_height, int n_frames) {
    return static_cast<uint8_t *>(mtb_host_alloc((size_t)image_width * image_height * 3 * (size_t)n_frames));
  }
  static uint8_t *AllocFrame(int image_width, int image_height) {
    return static_cast<uint8_t *>(mtb_host_alloc((size_t)image_width * image_height * 3));
  }
  static void FreeFrame(uint8_t *p) { mtb_host_free(p); }
  void SetMaxRecursionLevel(int level) { max_recursion_level = level; }
  void SetDevices(const std::vector<int> &devices) { scene.tree.SetDevices(devices); }
  void SetFlags(uint32_t flags) { scene.tree.SetFlags(flags); }
  mtb_stats last_stats{};

 private:
  bool RenderBatch(int image_width, int image_height, int samples_per_axis, const std::vector<Camera> &cams,
                   const std::vector<std::vector<Light>> *lights, uint8_t *out, bool synchronous) {
    if (!was_scene_finalized) {
      puts("Finalizing tree.");
      if (!scene.tree.Finalize(&scene.materials, &scene.textures)) return false;
      was_scene_finalized = true;
    }
    mtb_context *ctx = scene.tree.context();
    std::vector<mtb_camera> mcams;
    for (const Camera &c : cams) mcams.push_back(c.AsMtb());
    std::vector<Light> flat;
    int32_t n_lights = 0;
    if (lights == nullptr) {
      if (mtb_set_lights(ctx, reinterpret_cast<const mtb_light *>(scene.lights.data()), (int32_t)scene.lights.size()) != MTB_OK) {
        return false;
      }
    } else {
      if (lights->size() != cams.size()) {
        fprintf(stderr, "error: %zu light sets for %zu cameras (one per view)\n", lights->size(), cams.size());
        return false;
      }
      n_lights = lights->empty() ? 0 : (int32_t)lights->front().size();
      for (const std::vector<Light> &ls : *lights) {
        if ((int32_t)ls.size() != n_lights) {
          fputs("error: every view needs the same number of lights\n", stderr);
          return false;
        }
        flat.insert(flat.end(), ls.begin(), ls.end());
      }
      flat.resize(flat.size() + 1);  // (non-NULL even with no lights: n_lights = 0 is not "the scene's lights")
    }
    const mtb_light *lp = lights == nullptr ? nullptr : reinterpret_cast<const mtb_light *>(flat.data());
    mtb_stats stats;
    // (samples_per_axis = 1: mtb_render_batch_ss is mtb_render_batch)
    const int rc = synchronous ? mtb_render_batch_ss(ctx, mcams.data(), (int32_t)mcams.size(), lp, n_lights, image_width, image_height,
                                                     samples_per_axis, max_recursion_level, out, &stats)
                               : mtb_render_batch_ss_async(ctx, mcams.data(), (int32_t)mcams.size(), lp, n_lights, image_width,
                                                           image_height, samples_per_axis, max_recursion_level, out);
    if (rc != MTB_OK) {
      fprintf(stderr, "error: %s\n", mtb_last_error(ctx));
      return false;
    }
    if (synchronous) last_stats = stats;
    return true;
  }

  Scene scene;
  bool was_scene_finalized = false;
  int max_recursion_level = MAX_RECURSION_LEVEL;
};

}  // namespace raytracer
