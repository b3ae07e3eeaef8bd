// Batches into device memory through the C++ classes of include/mythtracer/: RayTraceBatchDevice.  Usage:
//   batch_device_check <scene.obj> <out_prefix> <w> <h> <s> <k>
// renders 2 output views of k sub-frames each (scene lights, depth 3; sub-frame j of view v turns the camera by
// 3 * v + 0.5 * j degrees of yaw) with s samples per axis into a cudaMalloc buffer, on a stream of its own and on the
// context's stream (nullptr), checks that both equal RayTraceBatch into host memory and that a host buffer is refused,
// then writes <out_prefix>.rgb (RGB24, the 2 output views, copied back from the device).
#include <cuda_runtime.h>

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
  if (argc < 7) return Fail("usage: batch_device_check <obj> <out_prefix> <w> <h> <s> <k>");
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

  const size_t bytes = 2 * (size_t)W * H * 3;
  std::vector<uint8_t> want(bytes), got(bytes), got_ctx(bytes);
  if (!mt.RayTraceBatch(W, H, S, K, cams, nullptr, want.data())) return Fail("RayTraceBatch");

  void *d_rgb = nullptr;
  cudaStream_t stream = nullptr;
  if (cudaMalloc(&d_rgb, bytes) != cudaSuccess || cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking) != cudaSuccess) {
    return Fail("cudaMalloc / cudaStreamCreate");
  }
  // on the caller's stream: a fill queued before the call is ordered before the batch, the copy queued after it sees it
  bool ok = cudaMemsetAsync(d_rgb, 0x5a, bytes, stream) == cudaSuccess && mt.RayTraceBatchDevice(W, H, S, K, cams, nullptr, d_rgb, stream) &&
            cudaMemcpyAsync(got.data(), d_rgb, bytes, cudaMemcpyDeviceToHost, stream) == cudaSuccess && cudaStreamSynchronize(stream) == cudaSuccess;
  if (!ok) return Fail("RayTraceBatchDevice on a stream");
  // on the context's own stream (nullptr): Wait() joins
  ok = cudaMemset(d_rgb, 0, bytes) == cudaSuccess && mt.RayTraceBatchDevice(W, H, S, K, cams, nullptr, d_rgb, nullptr) && mt.Wait() &&
       cudaMemcpy(got_ctx.data(), d_rgb, bytes, cudaMemcpyDeviceToHost) == cudaSuccess;
  if (!ok) return Fail("RayTraceBatchDevice on the context's stream");
  std::vector<uint8_t> host(bytes);
  const bool refused = !mt.RayTraceBatchDevice(W, H, S, K, cams, nullptr, host.data(), stream);
  cudaStreamDestroy(stream);
  cudaFree(d_rgb);
  if (got != want) return Fail("device batch on a stream != RayTraceBatch");
  if (got_ctx != want) return Fail("device batch on the context's stream != RayTraceBatch");
  if (!refused) return Fail("a host buffer was accepted as d_rgb");

  FILE *f = fopen((std::string(argv[2]) + ".rgb").c_str(), "wb");
  if (f == nullptr) return Fail("opening the output");
  const bool written = fwrite(got.data(), 1, got.size(), f) == got.size();
  if (fclose(f) != 0 || !written) return Fail("writing the output");
  puts("device ok");
  return 0;
}
