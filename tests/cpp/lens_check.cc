// Thin-lens batches through the C++ classes of include/mythtracer/: RayTraceBatch with lens samples.  Usage:
//   lens_check <scene.obj> <out_prefix> <w> <h> <s> <k>
// renders 2 output views of k sub-frames each (scene lights, depth 3; the sub-frames of view v share the camera turned
// by 3 * v degrees of yaw, sub-frame j takes lens point (4 cos(2 pi j / k), 4 sin(2 pi j / k)) focused at 150) with s
// samples per axis, checks that centred samples give the bytes of the pinhole overload, that a lens vector of the wrong
// length and a focus distance of 0 are refused, then writes <out_prefix>.rgb (RGB24, the 2 output views).
#include <cmath>
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
  if (argc < 7) return Fail("usage: lens_check <obj> <out_prefix> <w> <h> <s> <k>");
  const int W = atoi(argv[3]), H = atoi(argv[4]), S = atoi(argv[5]), K = atoi(argv[6]);
  MythTracer mt;
  if (!mt.LoadObj(argv[1])) return Fail("LoadObj");
  mt.SetMaxRecursionLevel(3);
  mt.GetScene()->lights.push_back(Light{{231.82174, 81.69966, 27.78259}, {0.3, 0.3, 0.3}, {1.0, 1.0, 1.0}, {1.0, 1.0, 1.0}});
  mt.GetScene()->lights.push_back(Light{{200, 95.0, 160}, {0.0, 0.0, 0.0}, {0.3, 0.3, 0.3}, {0.3, 0.3, 0.3}});
  std::vector<Camera> cams;
  std::vector<mtb_lens> lenses, centred;
  for (int v = 0; v < 2; v++) {
    for (int j = 0; j < K; j++) {
      cams.push_back(Camera{{301.37, 57.21, 161.13}, 4.0, 243.0 + 3.0 * v, 0.0, 110.0});
      const double a = 2.0 * M_PI * j / K;
      lenses.push_back(mtb_lens{4.0 * cos(a), 4.0 * sin(a), 150.0});
      centred.push_back(mtb_lens{0.0, 0.0, 150.0});
    }
  }

  const size_t frame_bytes = (size_t)W * H * 3;
  std::vector<uint8_t> rgb(2 * frame_bytes), a(2 * frame_bytes), b(2 * frame_bytes);
  if (!mt.RayTraceBatch(W, H, S, K, cams, lenses, nullptr, rgb.data())) return Fail("RayTraceBatch with lenses");
  if (!mt.RayTraceBatch(W, H, S, K, cams, centred, nullptr, a.data()) || !mt.RayTraceBatch(W, H, S, K, cams, nullptr, b.data())) {
    return Fail("RayTraceBatch with centred lenses / without lenses");
  }
  if (a != b) return Fail("centred lens samples != the pinhole batch");
  if (K > 1 && rgb == b) return Fail("an aperture gave the pinhole bytes");
  const std::vector<mtb_lens> short_list(lenses.begin(), lenses.end() - 1);
  if (mt.RayTraceBatch(W, H, S, K, cams, short_list, nullptr, a.data())) return Fail("a lens list shorter than the cameras was accepted");
  std::vector<mtb_lens> unfocused = lenses;
  unfocused[0].focus_distance = 0.0;
  if (mt.RayTraceBatch(W, H, S, K, cams, unfocused, nullptr, a.data())) return Fail("focus_distance 0 was accepted");

  FILE *f = fopen((std::string(argv[2]) + ".rgb").c_str(), "wb");
  if (f == nullptr) return Fail("opening the output");
  const bool ok = fwrite(rgb.data(), 1, rgb.size(), f) == rgb.size();
  if (fclose(f) != 0 || !ok) return Fail("writing the output");
  puts("lens ok");
  return 0;
}
