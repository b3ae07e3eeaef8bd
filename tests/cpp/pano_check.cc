// Panorama batches through the C++ classes of include/mythtracer/: RayTraceBatch with panorama parameters.  Usage:
//   pano_check <scene.obj> <out_prefix> <w> <h> <s> <k>
// renders 2 output views of k sub-frames each (scene lights, depth 3; the sub-frames of view v share the camera turned
// by 3 * v degrees of yaw, and view 0 is the left eye (-3.2), view 1 the right eye (+3.2) of a full 360 x 180 panorama)
// with s samples per axis, checks that an empty eye-offset list gives the bytes of all-zero offsets, that an eye-offset
// list of the wrong length, an h_fov of 0 and a v_fov above 180 are refused, then writes <out_prefix>.rgb (RGB24, the
// 2 output views).
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
  if (argc < 7) return Fail("usage: pano_check <obj> <out_prefix> <w> <h> <s> <k>");
  const int W = atoi(argv[3]), H = atoi(argv[4]), S = atoi(argv[5]), K = atoi(argv[6]);
  MythTracer mt;
  if (!mt.LoadObj(argv[1])) return Fail("LoadObj");
  mt.SetMaxRecursionLevel(3);
  mt.GetScene()->lights.push_back(Light{{231.82174, 81.69966, 27.78259}, {0.3, 0.3, 0.3}, {1.0, 1.0, 1.0}, {1.0, 1.0, 1.0}});
  mt.GetScene()->lights.push_back(Light{{200, 95.0, 160}, {0.0, 0.0, 0.0}, {0.3, 0.3, 0.3}, {0.3, 0.3, 0.3}});
  std::vector<Camera> cams;
  std::vector<double> eyes, zeros;
  for (int v = 0; v < 2; v++) {
    for (int j = 0; j < K; j++) {
      cams.push_back(Camera{{301.37, 57.21, 161.13}, 4.0, 243.0 + 3.0 * v, 0.0, 110.0});
      eyes.push_back(v == 0 ? -3.2 : 3.2);
      zeros.push_back(0.0);
    }
  }

  const size_t frame_bytes = (size_t)W * H * 3;
  std::vector<uint8_t> rgb(2 * frame_bytes), a(2 * frame_bytes), b(2 * frame_bytes);
  if (!mt.RayTraceBatch(W, H, S, K, cams, 360.0, 180.0, eyes, nullptr, rgb.data())) return Fail("RayTraceBatch with a panorama");
  if (!mt.RayTraceBatch(W, H, S, K, cams, 360.0, 180.0, zeros, nullptr, a.data()) ||
      !mt.RayTraceBatch(W, H, S, K, cams, 360.0, 180.0, std::vector<double>(), nullptr, b.data())) {
    return Fail("RayTraceBatch with zero / no eye offsets");
  }
  if (a != b) return Fail("an empty eye-offset list != all-zero offsets");
  if (rgb == a) return Fail("the eye offsets changed nothing");
  const std::vector<double> short_list(eyes.begin(), eyes.end() - 1);
  if (mt.RayTraceBatch(W, H, S, K, cams, 360.0, 180.0, short_list, nullptr, a.data())) return Fail("an eye-offset list shorter than the cameras was accepted");
  if (mt.RayTraceBatch(W, H, S, K, cams, 0.0, 180.0, eyes, nullptr, a.data())) return Fail("h_fov 0 was accepted");
  if (mt.RayTraceBatch(W, H, S, K, cams, 360.0, 180.5, eyes, nullptr, a.data())) return Fail("v_fov 180.5 was accepted");

  FILE *f = fopen((std::string(argv[2]) + ".rgb").c_str(), "wb");
  if (f == nullptr) return Fail("opening the output");
  const bool ok = fwrite(rgb.data(), 1, rgb.size(), f) == rgb.size();
  if (fclose(f) != 0 || !ok) return Fail("writing the output");
  puts("pano ok");
  return 0;
}
