// Host-side CUDA helpers shared by the engine (engine.cu), the R1CS checker (r1cs.cu), the device input parser
// (inputs.cu), the NTT (ntt.cu) and the C ABI (capi.cpp).  The functions are defined in cuda_util.cpp.
#pragma once
#include <cuda_runtime.h>

#include <functional>
#include <string>

#include "graph.hpp"

namespace gw {

static const char* const NO_DEVICE_ERROR = "no CUDA device available: this library has no CPU fallback";

// The library works on the device it is told to, and leaves the calling thread's current device as it found it
// (a caller that mixes this library with its own CUDA code must not find itself on another GPU after a call).
struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int device) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) throw Error(std::string("CUDA error: ") + cudaGetErrorString(e) + " at cudaSetDevice");
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
  DeviceGuard(const DeviceGuard&) = delete;
};

#define CUDA_CHECK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) throw Error(std::string("CUDA error: ") + cudaGetErrorString(e_) + " at " #x); } while (0)

// no copy may still target the caller's (or a pinned ring's) memory when a host-buffer call returns, also on errors
struct StreamDrain {
  cudaStream_t a, b;
  ~StreamDrain() { if (a) cudaStreamSynchronize(a); if (b) cudaStreamSynchronize(b); }
};

// visible CUDA devices; 0 when the runtime cannot count them
int cuda_device_count();
// throws NO_DEVICE_ERROR when no device is visible, and "CUDA device index out of range" unless `device` is one of them
void check_device(int device);
// B independent items over n_gpus devices starting at first_device, no collective: shard g = [B g / n_gpus, B (g + 1) / n_gpus)
// runs fn(first_device + g, lo, hi) on a thread of its own, pinned near its GPU.  Every thread is joined; then the first
// error in shard order is rethrown.
void run_shards(size_t B, int n_gpus, int first_device, const std::function<void(int, size_t, size_t)>& fn);

}  // namespace gw
