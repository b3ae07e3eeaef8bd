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
    return RenderBatch(image_width, image_height, 1, 1, cams, lights, out, nullptr, true);
  }
  bool RayTraceBatchAsync(int image_width, int image_height, const std::vector<Camera> &cams, const std::vector<std::vector<Light>> *lights,
                          uint8_t *pinned_out) {
    return RenderBatch(image_width, image_height, 1, 1, cams, lights, pinned_out, nullptr, false);
  }
  // Anti-aliased batches (mtb_render_batch_ss): samples_per_axis s = 1, 2, 4 or 8; every output pixel is the rounded
  // mean of the s x s pixels of the same view rendered at (s*w) x (s*h).  `out` holds cams.size() * w * h * 3 bytes.
  bool RayTraceBatch(int image_width, int image_height, int samples_per_axis, const std::vector<Camera> &cams,
                     const std::vector<std::vector<Light>> *lights, uint8_t *out) {
    return RenderBatch(image_width, image_height, samples_per_axis, 1, cams, lights, out, nullptr, true);
  }
  bool RayTraceBatchAsync(int image_width, int image_height, int samples_per_axis, const std::vector<Camera> &cams,
                          const std::vector<std::vector<Light>> *lights, uint8_t *pinned_out) {
    return RenderBatch(image_width, image_height, samples_per_axis, 1, cams, lights, pinned_out, nullptr, false);
  }
  // The same batch with the batch form of WorkChunk::output_debug (mtb_render_batch_debug): *debug_out is resized to
  // cams.size() * (s*h) * (s*w) entries, view-major, the primary hit of every sample of every view (for s = 1, of every
  // pixel): entry (x, y) of view v is what RayTrace(WorkChunk*) leaves for pixel (x, y) of an (s*w) x (s*h) frame.
  bool RayTraceBatch(int image_width, int image_height, int samples_per_axis, const std::vector<Camera> &cams,
                     const std::vector<std::vector<Light>> *lights, uint8_t *out, std::vector<PerPixelDebugInfo> *debug_out) {
    // (other sizes are refused by the call before it writes anything; debug_out == nullptr: the overload above)
    mtb_debug *dbg = nullptr;
    if (debug_out != nullptr && (samples_per_axis == 1 || samples_per_axis == 2 || samples_per_axis == 4 || samples_per_axis == 8) &&
        image_width > 0 && image_height > 0) {
      debug_out->resize(cams.size() * (size_t)(samples_per_axis * image_height) * (size_t)(samples_per_axis * image_width));
      dbg = reinterpret_cast<mtb_debug *>(debug_out->data());
    }
    return RenderBatch(image_width, image_height, samples_per_axis, 1, cams, lights, out, dbg, true);
  }
  // Accumulated batches (mtb_render_batch_accum): every output view is the rounded mean of all subframes * s * s
  // samples of its `subframes` sub-frames (motion blur: a camera path over the shutter interval; soft shadows: jittered
  // positions on an area light).  cams (and *lights) hold `subframes` entries per output view, output-major; `out` holds
  // cams.size() / subframes * w * h * 3 bytes.  subframes = 1: the overloads above.
  bool RayTraceBatch(int image_width, int image_height, int samples_per_axis, int subframes, const std::vector<Camera> &cams,
                     const std::vector<std::vector<Light>> *lights, uint8_t *out) {
    return RenderBatch(image_width, image_height, samples_per_axis, subframes, cams, lights, out, nullptr, true);
  }
  bool RayTraceBatchAsync(int image_width, int image_height, int samples_per_axis, int subframes, const std::vector<Camera> &cams,
                          const std::vector<std::vector<Light>> *lights, uint8_t *pinned_out) {
    return RenderBatch(image_width, image_height, samples_per_axis, subframes, cams, lights, pinned_out, nullptr, false);
  }
  // Batches left in device memory (mtb_render_batch_device): the bytes of the overloads above, written to d_rgb, DEVICE
  // memory of the context's device 0 (cams.size() / subframes * w * h * 3 bytes), and ordered on `stream` (a
  // cudaStream_t of device 0; nullptr = the context's own stream): the batch starts after the work queued there before
  // the call, and work queued there afterwards sees the frames.  Returns once the work is queued.  RGB only: the planes
  // of a batch in device memory come from the C ABI.
  bool RayTraceBatchDevice(int image_width, int image_height, int samples_per_axis, int subframes, const std::vector<Camera> &cams,
                           const std::vector<std::vector<Light>> *lights, void *d_rgb, void *stream) {
    return RenderBatch(image_width, image_height, samples_per_axis, subframes, cams, lights, static_cast<uint8_t *>(d_rgb), nullptr, false,
                       true, stream);
  }
  // Depth of field (mtb_render_batch_lens): the accumulated batch above with one thin-lens sample (u, v,
  // focus_distance) per camera.  Camera i's primary rays start at its origin moved by u along the image's right and v
  // along its down direction, and pass through the points where its pinhole rays meet the focal plane at
  // focus_distance; k lens points spread over an aperture, averaged as sub-frames, give depth of field.  A centred
  // sample (0, 0, f) is the pinhole ray.  lenses.size() must equal cams.size().
  bool RayTraceBatch(int image_width, int image_height, int samples_per_axis, int subframes, const std::vector<Camera> &cams,
                     const std::vector<mtb_lens> &lenses, const std::vector<std::vector<Light>> *lights, uint8_t *out) {
    if (lenses.size() != cams.size()) {
      fprintf(stderr, "error: %zu lens samples for %zu cameras (one per camera)\n", lenses.size(), cams.size());
      return false;
    }
    return RenderBatch(image_width, image_height, samples_per_axis, subframes, cams, lights, out, nullptr, true, false, nullptr, lenses.data());
  }
  // Panoramas (mtb_render_batch_pano): the accumulated batch above with every camera rendering an h_fov x v_fov degree
  // longitude / latitude grid around its origin, turned by its pitch, yaw and roll (its aov is ignored); (360, 180) is a
  // full equirectangular panorama.  eye_offsets: empty (all 0) or one per camera, the distance each column's origin
  // moves along its tangent; -IPD/2 and +IPD/2 give the two eyes of an omni-directional stereo pair.
  bool RayTraceBatch(int image_width, int image_height, int samples_per_axis, int subframes, const std::vector<Camera> &cams, double h_fov,
                     double v_fov, const std::vector<double> &eye_offsets, const std::vector<std::vector<Light>> *lights, uint8_t *out) {
    if (!eye_offsets.empty() && eye_offsets.size() != cams.size()) {
      fprintf(stderr, "error: %zu eye offsets for %zu cameras (one per camera, or none)\n", eye_offsets.size(), cams.size());
      return false;
    }
    const Panorama pano{h_fov, v_fov, eye_offsets.empty() ? nullptr : eye_offsets.data()};
    return RenderBatch(image_width, image_height, samples_per_axis, subframes, cams, lights, out, nullptr, true, false, nullptr, nullptr, &pano);
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
  struct Panorama {
    double h_fov, v_fov;
    const double *eye_offsets;
  };
  bool RenderBatch(int image_width, int image_height, int samples_per_axis, int subframes, const std::vector<Camera> &cams,
                   const std::vector<std::vector<Light>> *lights, uint8_t *out, mtb_debug *dbg, bool synchronous, bool device = false,
                   void *stream = nullptr, const mtb_lens *lenses = nullptr, const Panorama *pano = nullptr) {
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
    int rc;
    if (subframes != 1 || device || lenses != nullptr || pano != nullptr) {
      if (subframes < 1 || cams.size() % (size_t)subframes != 0) {
        fprintf(stderr, "error: %zu cameras are not a whole number of output views of %d subframes\n", cams.size(), subframes);
        return false;
      }
      const int32_t n_out = (int32_t)(cams.size() / (size_t)subframes);
      if (lenses != nullptr) {
        rc = mtb_render_batch_lens(ctx, mcams.data(), lenses, n_out, subframes, lp, n_lights, image_width, image_height, samples_per_axis,
                                   max_recursion_level, out, nullptr, nullptr, &stats);
      } else if (pano != nullptr) {
        rc = mtb_render_batch_pano(ctx, mcams.data(), pano->eye_offsets, n_out, subframes, pano->h_fov, pano->v_fov, lp, n_lights, image_width,
                                   image_height, samples_per_axis, max_recursion_level, out, nullptr, nullptr, &stats);
      } else if (device) {
        rc = mtb_render_batch_device(ctx, mcams.data(), n_out, subframes, lp, n_lights, image_width, image_height, samples_per_axis,
                                     max_recursion_level, out, nullptr, nullptr, stream, nullptr);
      } else {
        rc = synchronous ? mtb_render_batch_accum(ctx, mcams.data(), n_out, subframes, lp, n_lights, image_width, image_height, samples_per_axis,
                                                  max_recursion_level, out, &stats)
                         : mtb_render_batch_accum_async(ctx, mcams.data(), n_out, subframes, lp, n_lights, image_width, image_height,
                                                        samples_per_axis, max_recursion_level, out);
      }
    } else {
      // (samples_per_axis = 1: mtb_render_batch_ss is mtb_render_batch; dbg = NULL: mtb_render_batch_debug is mtb_render_batch_ss)
      rc = synchronous ? mtb_render_batch_debug(ctx, mcams.data(), (int32_t)mcams.size(), lp, n_lights, image_width, image_height,
                                                samples_per_axis, max_recursion_level, out, dbg, nullptr, &stats)
                       : mtb_render_batch_ss_async(ctx, mcams.data(), (int32_t)mcams.size(), lp, n_lights, image_width, image_height,
                                                   samples_per_axis, max_recursion_level, out);
    }
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
