// The reference's single-process animation driver (VerStarting/main_local.cc:24-155) on the B200 renderer
// (SURVEY.md section 8 f3): orbiting camera, lights re-set every frame, raw RGB24 frames to
// anim/dump_%05i.raw.  The model path, resolution and frame range are arguments instead of constants.
//
//   mythtracer_local_b200 scene.obj [width height first_frame last_frame out_dir frames_per_call samples_per_axis]
//
// frames_per_call N > 1 renders N consecutive frames per batch call (one launch for all of them: a 480x270 frame alone
// is less than one wave of the B200); the files and their bytes are the same as with N = 1, the default.
// samples_per_axis s = 2, 4 or 8 writes anti-aliased frames (s x s samples per pixel, averaged on the device) of the
// same width x height; they always go through the batch path, with N frames per call.  s = 1, the default, is the
// reference's one ray per pixel.
#include <sys/stat.h>
#include <sys/types.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include <mythtracer/mythtracer.h>

using raytracer::AABB;
using raytracer::Camera;
using raytracer::Light;
using raytracer::MythTracer;

namespace {

// main_local.cc:72-76
Camera OrbitCamera(double angle) { return Camera{{300.0, 107.0, 40.0}, 30.0, angle + 90, 0.0, 110.0}; }

// main_local.cc:79-110
void SetRig(MythTracer &mt) {
  auto &lights = mt.GetScene()->lights;
  lights.clear();
  lights.push_back(Light{{231.82174, 81.69966, -27.78259}, {0.3, 0.3, 0.3}, {1.0, 1.0, 1.0}, {1.0, 1.0, 1.0}});
  for (double z : {0.0, 80.0, 160.0}) lights.push_back(Light{{200, 80.0, z}, {0.0, 0.0, 0.0}, {0.3, 0.3, 0.3}, {0.3, 0.3, 0.3}});
}

bool WriteFrame(const char *out_dir, int number, const uint8_t *pixels, size_t frame_bytes) {
  puts("Writing");
  char fname[512];
  snprintf(fname, sizeof(fname), "%s/dump_%.5i.raw", out_dir, number);
  FILE *f = fopen(fname, "wb");
  if (f == nullptr) return false;
  fwrite(pixels, frame_bytes, 1, f);
  fclose(f);
  return true;
}

// frames_per_call > 1: `per_call` consecutive frames per batch call (the last batch may be partial), into two pinned
// batch buffers in rotation: batch k is written to disk while batch k+1 renders.  Every frame uses the same rig, so
// the views take the scene's lights.
int RenderBatches(MythTracer &mt, int W, int H, int first, int last, const char *out_dir, int per_call, int samples_per_axis) {
  SetRig(mt);
  std::vector<int> numbers;
  std::vector<Camera> cams;
  int frame = 0;
  for (double angle = 0.0; angle <= 360.0; angle += 2.0, frame++) {
    if (frame < first || frame > last) continue;
    numbers.push_back(frame);
    cams.push_back(OrbitCamera(angle));
  }
  uint8_t *bufs[2] = {MythTracer::AllocFrames(W, H, per_call), MythTracer::AllocFrames(W, H, per_call)};
  if (bufs[0] == nullptr || bufs[1] == nullptr) return 1;
  const size_t frame_bytes = (size_t)W * H * 3;
  auto write_batch = [&](size_t begin, size_t count, const uint8_t *pixels) {
    for (size_t i = 0; i < count; i++) {
      if (!WriteFrame(out_dir, numbers[begin + i], pixels + i * frame_bytes, frame_bytes)) return false;
    }
    return true;
  };
  const auto t0 = std::chrono::steady_clock::now();
  size_t pending_begin = 0, pending_count = 0;
  int calls = 0;
  for (size_t begin = 0; begin < cams.size(); begin += (size_t)per_call, calls++) {
    const size_t count = std::min(cams.size() - begin, (size_t)per_call);
    const std::vector<Camera> batch(cams.begin() + (long)begin, cams.begin() + (long)(begin + count));
    printf("Rendering %zu frames.\n", count);
    if (!mt.RayTraceBatchAsync(W, H, samples_per_axis, batch, nullptr, bufs[calls & 1])) return 1;
    if (pending_count > 0 && !write_batch(pending_begin, pending_count, bufs[(calls + 1) & 1])) return 1;  // overlaps the render
    if (!mt.Wait()) return 1;
    pending_begin = begin;
    pending_count = count;
  }
  if (pending_count > 0 && !write_batch(pending_begin, pending_count, bufs[(calls + 1) & 1])) return 1;
  const double total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  MythTracer::FreeFrame(bufs[0]);
  MythTracer::FreeFrame(bufs[1]);
  const size_t n = cams.size();
  printf("Done: %zu frames in %d calls, %.2f ms per frame (render + copies + file writes, double-buffered)\n", n, calls,
         n ? total_ms / (double)n : 0.0);
  return 0;
}

}  // namespace

int main(int argc, char **argv) {
  if (argc < 2) {
    puts("usage: mythtracer_local_b200 scene.obj [width height first_frame last_frame out_dir frames_per_call samples_per_axis]");
    return 1;
  }
  const int W = argc > 2 ? atoi(argv[2]) : 1920 / 4, H = argc > 3 ? atoi(argv[3]) : 1080 / 4;
  const int first = argc > 4 ? atoi(argv[4]) : 74, last = argc > 5 ? atoi(argv[5]) : 180;
  const char *out_dir = argc > 6 ? argv[6] : "anim";
  const int per_call = argc > 7 ? atoi(argv[7]) : 1;
  const int samples = argc > 8 ? atoi(argv[8]) : 1;
  if (per_call < 1) {
    puts("frames_per_call must be >= 1");
    return 1;
  }
  if (samples != 1 && samples != 2 && samples != 4 && samples != 8) {
    puts("samples_per_axis must be 1, 2, 4 or 8");
    return 1;
  }
  printf("Creating %s/ directory\n", out_dir);
  mkdir(out_dir, 0700);
  printf("Resolution: %u %u\n", W, H);

  MythTracer mt;
  if (!mt.LoadObj(argv[1])) return 1;
  const AABB aabb = mt.GetScene()->tree.GetAABB();
  printf("%f %f %f x %f %f %f\n", aabb.min.v[0], aabb.min.v[1], aabb.min.v[2], aabb.max.v[0], aabb.max.v[1], aabb.max.v[2]);

  if (per_call > 1 || samples > 1) return RenderBatches(mt, W, H, first, last, out_dir, per_call, samples);

  // Two pinned frames in rotation: while frame k+1 renders (queued without waiting), frame k is written to disk.
  uint8_t *frames[2] = {MythTracer::AllocFrame(W, H), MythTracer::AllocFrame(W, H)};
  if (frames[0] == nullptr || frames[1] == nullptr) return 1;
  const size_t frame_bytes = (size_t)W * H * 3;
  auto write_frame = [&](int number, const uint8_t *pixels) { return WriteFrame(out_dir, number, pixels, frame_bytes); };
  int frame = 0;
  int rendered = 0, pending = -1;
  const auto t0 = std::chrono::steady_clock::now();
  for (double angle = 0.0; angle <= 360.0; angle += 2.0, frame++) {
    if (frame < first || frame > last) continue;
    Camera cam = OrbitCamera(angle);
    SetRig(mt);
    puts("Rendering.");
    if (!mt.RayTraceAsync(W, H, &cam, frames[rendered & 1])) return 1;
    if (pending >= 0 && !write_frame(pending, frames[(rendered + 1) & 1])) return 1;  // overlaps the render
    if (!mt.Wait()) return 1;
    pending = frame;
    rendered++;
  }
  if (pending >= 0 && !write_frame(pending, frames[(rendered + 1) & 1])) return 1;
  const double total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  MythTracer::FreeFrame(frames[0]);
  MythTracer::FreeFrame(frames[1]);
  printf("Done: %d frames, %.2f ms per frame (render + copies + file writes, double-buffered)\n", rendered, rendered ? total_ms / rendered : 0.0);
  return 0;
}
