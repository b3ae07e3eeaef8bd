// Accumulated batches through the C++ classes of include/mythtracer/: RayTraceBatch / RayTraceBatchAsync with
// `subframes`.  Usage:
//   accum_check <scene.obj> <out_prefix> <w> <h> <s> <k>
// renders 2 output views of k sub-frames each (scene lights, depth 3; sub-frame j of view v turns the camera by
// 3 * v + 0.5 * j degrees of yaw) with s samples per axis, checks that the asynchronous call gives the bytes of the
// synchronous one, that subframes = 1 gives the bytes of the overload without it and that a camera count that is not a
// multiple of k is refused, then writes <out_prefix>.rgb (RGB24, the 2 output views).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

#include <mythtracer/mythtracer.h>

using raytracer::Camera;
using raytracer::Light;
using raytracer::MythTracer;

static int Fail(const char *what) {
  fprintf(stderr, "FAIL: %s\n", what);
  return 1;
}

int main(int argc, char **argv) {
  if (argc < 7) return Fail("usage: accum_check <obj> <out_prefix> <w> <h> <s> <k>");
  const int W = atoi(argv[3]), H = atoi(argv[4]), S = atoi(argv[5]), K = atoi(argv[6]);
  MythTracer mt;
  if (!mt.LoadObj(argv[1])) return Fail("LoadObj");
  mt.SetMaxRecursionLevel(3);
  mt.GetScene()->lights.push_back(Light{{231.82174, 81.69966, 27.78259}, {0.3, 0.3, 0.3}, {1.0, 1.0, 1.0}, {1.0, 1.0, 1.0}});
  mt.GetScene()->lights.push_back(Light{{200, 95.0, 160}, {0.0, 0.0, 0.0}, {0.3, 0.3, 0.3}, {0.3, 0.3, 0.3}});
  std::vector<Camera> cams;
  for (int v = 0; v < 2; v++) {
    for (int j = 0; j < K; j++) cams.push_back(Camera{{301.37, 57.21, 161.13}, 4.0, 243.0 + 3.0 * v + 0.5 * j, 0.0, 110.0});
  }

  const size_t frame_bytes = (size_t)W * H * 3;
  std::vector<uint8_t> rgb(2 * frame_bytes);
  if (!mt.RayTraceBatch(W, H, S, K, cams, nullptr, rgb.data())) return Fail("RayTraceBatch with subframes");
  uint8_t *pinned = MythTracer::AllocFrames(W, H, 2);
  if (pinned == nullptr) return Fail("AllocFrames");
  memset(pinned, 0, 2 * frame_bytes);
  const bool queued = mt.RayTraceBatchAsync(W, H, S, K, cams, nullptr, pinned) && mt.Wait();
  const bool same = queued && memcmp(pinned, rgb.data(), rgb.size()) == 0;
  MythTracer::FreeFrame(pinned);
  if (!queued) return Fail("RayTraceBatchAsync with subframes");
  if (!same) return Fail("asynchronous accumulated batch != synchronous one");

  const std::vector<Camera> two(cams.begin(), cams.begin() + 2);
  std::vector<uint8_t> a(2 * frame_bytes), b(2 * frame_bytes);
  if (!mt.RayTraceBatch(W, H, S, 1, two, nullptr, a.data()) || !mt.RayTraceBatch(W, H, S, two, nullptr, b.data())) {
    return Fail("RayTraceBatch with subframes = 1");
  }
  if (a != b) return Fail("subframes = 1 != the overload without subframes");
  if (K > 1) {
    const std::vector<Camera> odd(cams.begin(), cams.begin() + K + 1);
    if (mt.RayTraceBatch(W, H, S, K, odd, nullptr, a.data())) return Fail("k + 1 cameras for subframes = k were accepted");
  }

  FILE *f = fopen((std::string(argv[2]) + ".rgb").c_str(), "wb");
  if (f == nullptr) return Fail("opening the output");
  const bool ok = fwrite(rgb.data(), 1, rgb.size(), f) == rgb.size();
  if (fclose(f) != 0 || !ok) return Fail("writing the output");
  puts("accum ok");
  return 0;
}
