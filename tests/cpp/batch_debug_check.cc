// The batch form of WorkChunk::output_debug through the C++ classes of include/mythtracer/: RayTraceBatch with a
// std::vector<PerPixelDebugInfo> output.  Usage:
//   batch_debug_check <scene.obj> <out_prefix> <w> <h> <s>
// renders 3 views (scene lights, depth 3) with s samples per axis, checks the vector's size, that the RGB equals the
// overload without debug output and that view 1's planes equal RayTrace(WorkChunk*) of an (s*w) x (s*h) frame, then
// writes <out_prefix>.rgb (RGB24) and <out_prefix>.dbg (32-byte PerPixelDebugInfo records), both view-major.
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include <mythtracer/mythtracer.h>

using raytracer::Camera;
using raytracer::Light;
using raytracer::MythTracer;
using raytracer::PerPixelDebugInfo;
using raytracer::WorkChunk;

static int Fail(const char *what) {
  fprintf(stderr, "FAIL: %s\n", what);
  return 1;
}

static bool Write(const char *prefix, const char *ext, const void *data, size_t bytes) {
  char path[4096];
  snprintf(path, sizeof(path), "%s%s", prefix, ext);
  FILE *f = fopen(path, "wb");
  if (f == nullptr) return false;
  const bool ok = fwrite(data, 1, bytes, f) == bytes;
  return fclose(f) == 0 && ok;
}

int main(int argc, char **argv) {
  if (argc < 6) return Fail("usage: batch_debug_check <obj> <out_prefix> <w> <h> <s>");
  const int W = atoi(argv[3]), H = atoi(argv[4]), S = atoi(argv[5]);
  MythTracer mt;
  if (!mt.LoadObj(argv[1])) return Fail("LoadObj");
  mt.SetMaxRecursionLevel(3);
  mt.GetScene()->lights.push_back(Light{{231.82174, 81.69966, 27.78259}, {0.3, 0.3, 0.3}, {1.0, 1.0, 1.0}, {1.0, 1.0, 1.0}});
  mt.GetScene()->lights.push_back(Light{{200, 95.0, 160}, {0.0, 0.0, 0.0}, {0.3, 0.3, 0.3}, {0.3, 0.3, 0.3}});
  std::vector<Camera> cams;
  for (int v = 0; v < 3; v++) cams.push_back(Camera{{301.37, 57.21, 161.13}, 4.0, 243.0 + 3.0 * v, 0.0, 110.0});

  const size_t per_view = (size_t)(S * W) * (size_t)(S * H);
  std::vector<uint8_t> rgb(cams.size() * W * H * 3), plain(rgb.size());
  std::vector<PerPixelDebugInfo> dbg(5);  // resized by the call
  if (!mt.RayTraceBatch(W, H, S, cams, nullptr, rgb.data(), &dbg)) return Fail("RayTraceBatch with debug_out");
  if (dbg.size() != cams.size() * per_view) return Fail("debug_out size");
  if (!mt.RayTraceBatch(W, H, S, cams, nullptr, plain.data())) return Fail("RayTraceBatch");
  if (plain != rgb) return Fail("RGB with debug_out != RGB without");

  WorkChunk chunk{S * W, S * H, 0, 0, S * W, S * H, cams[1], {}, {}};
  chunk.output_bitmap.resize(per_view * 3);
  chunk.output_debug.resize(per_view);
  if (!mt.RayTrace(&chunk)) return Fail("RayTrace(WorkChunk*)");
  if (memcmp(chunk.output_debug.data(), dbg.data() + per_view, per_view * sizeof(PerPixelDebugInfo)) != 0) {
    return Fail("view 1 != RayTrace(WorkChunk*) output_debug");
  }
  if (!Write(argv[2], ".rgb", rgb.data(), rgb.size()) || !Write(argv[2], ".dbg", dbg.data(), dbg.size() * sizeof(PerPixelDebugInfo))) {
    return Fail("writing the outputs");
  }
  puts("batch debug ok");
  return 0;
}
