// Host-side CUDA helpers shared by the engine (engine.cu) and the R1CS checker (r1cs.cu).
#pragma once
#include <cuda_runtime.h>

#include <string>

#include "graph.hpp"

namespace gw {

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

// pins the calling thread to the CPUs of the NUMA node of `device` (engine.cu; GW_NUMA=0 turns it off)
void bind_thread_near_device(int device);

}  // namespace gw
