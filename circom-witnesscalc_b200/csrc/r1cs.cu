// R1CS check of witness rows on sm_100a: for every row, the lowest constraint k with <A_k,w> * <B_k,w> != <C_k,w>.
//
// Execution model: one thread = one witness row, so the 32 lanes of a warp check 32 rows against the SAME constraint
// stream (warp-uniform control flow, no divergence).  Each warp streams the 8-byte program items itself, as
// eval_batch_kernel streams its instruction slots: lane l loads item base + l (one coalesced 256-byte read), two
// blocks of 32 are staged in the warp's ring in shared memory, the next block waits in a register, and every lane
// reads the current item from shared memory (a broadcast).  The most used constants are staged in shared memory
// once per CTA.  A term reads the 32 bytes of its wire from the lane's own row: two 16-byte loads of one sector.
// Persistent CTAs (one per SM) walk tiles of rows; a warp whose 32 rows have all failed stops early.
#include <cuda_runtime.h>

#include <algorithm>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "cuda_util.hpp"
#include "r1cs.hpp"
#include "r1cs_eval.cuh"

namespace gw {

namespace {

struct RParams {
  const uint2* code; uint32_t n_items;
  const uint4* consts; uint32_t n_hot;     // the first n_hot table constants are staged in shared memory
  const uint8_t* witness; unsigned long long pitch, B;
  uint32_t n_constraints, n_tiles;
  uint32_t* first_failed;
};

const int R1_RING = 64;                  // program items staged per warp (two blocks of 32)
const int R1_MAX_THREADS = 512;          // one persistent CTA per SM; 512 threads x 128 registers = the register file

}  // namespace

// Dynamic shared memory: [n_hot][2] hot constants (uint4) | [T/32 warps][R1_RING] program items (uint2).
__global__ void __launch_bounds__(R1_MAX_THREADS, 1) r1cs_check_kernel(const RParams p) {
  extern __shared__ uint4 smem[];
  const int T = blockDim.x;
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const uint4* hot = smem;
  uint2* ring = reinterpret_cast<uint2*>(smem + 2 * (size_t)p.n_hot) + (tid >> 5) * R1_RING;
  const uint32_t n = p.n_items;

  for (uint32_t k = tid; k < 2 * p.n_hot; k += T) smem[k] = __ldg(p.consts + k);
  __syncthreads();

  auto const_val = [&](uint32_t c) {
    fe r;
    const uint4 lo = c < p.n_hot ? hot[2 * c] : __ldg(p.consts + 2 * (size_t)c);
    const uint4 hi = c < p.n_hot ? hot[2 * c + 1] : __ldg(p.consts + 2 * (size_t)c + 1);
    r.l[0] = lo.x; r.l[1] = lo.y; r.l[2] = lo.z; r.l[3] = lo.w; r.l[4] = hi.x; r.l[5] = hi.y; r.l[6] = hi.z; r.l[7] = hi.w;
    return r;
  };

  for (uint32_t tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
    const unsigned long long row = (unsigned long long)tile * T + tid;
    const bool active = row < p.B;
    if (__all_sync(0xFFFFFFFFu, !active)) continue;
    const uint4* w = reinterpret_cast<const uint4*>(p.witness + (active ? row : p.B - 1) * p.pitch);
    auto wire_val = [&](uint32_t i) {
      fe r;
      const uint4 lo = __ldg(w + 2 * (size_t)i), hi = __ldg(w + 2 * (size_t)i + 1);
      r.l[0] = lo.x; r.l[1] = lo.y; r.l[2] = lo.z; r.l[3] = lo.w; r.l[4] = hi.x; r.l[5] = hi.y; r.l[6] = hi.z; r.l[7] = hi.w;
      return r;
    };

    // ring: blocks 0 and 1 staged, block 2 in flight in nblk
    __syncwarp();
    ring[lane] = __ldg(p.code + min((uint32_t)lane, n - 1));
    ring[32 + lane] = __ldg(p.code + min(32u + lane, n - 1));
    uint2 nblk = __ldg(p.code + min(64u + lane, n - 1));
    __syncwarp();
    uint32_t pc = 0;
    auto next = [&](uint32_t& a, uint32_t& b) {
      const uint2 it = ring[pc & (R1_RING - 1)];
      a = it.x; b = it.y;
      pc++;
      if ((pc & 31u) == 0) {
        // block (pc >> 5) - 1 is consumed: stage block (pc >> 5) + 1 in its half, start loading the one after it
        __syncwarp();
        ring[(((pc >> 5) - 1) & 1u) * 32u + lane] = nblk;
        nblk = __ldg(p.code + min(((pc >> 5) + 2u) * 32u + lane, n - 1));
        __syncwarp();
      }
    };

    uint32_t first = R1CS_OK;
#pragma unroll 1
    for (uint32_t k = 0; k < p.n_constraints; k++) {
      uint32_t na, nb, nc, unused;
      next(na, nb);
      next(nc, unused);
      bool bad = false;
      fe a, b, c;
#pragma unroll 1
      for (int which = 0; which < 3; which++) {   // one copy of the term loop for A, B and C
        const fe v = r1cs_lc(which == 0 ? na : which == 1 ? nb : nc, next, wire_val, const_val, &bad);
        if (which == 0) a = v; else if (which == 1) b = v; else c = v;
      }
      if (first == R1CS_OK && (bad || !r1cs_holds(a, b, c))) first = k;
      if (__all_sync(0xFFFFFFFFu, first != R1CS_OK || !active)) break;
    }
    if (active) p.first_failed[row] = first;
  }
}

struct R1cs::Dev {
  int device = -1;
  int sms = 0;
  size_t smem_max = 0;
  uint2* code = nullptr; uint4* consts = nullptr;
  // staging of the host-row entry point: two chunks of dense rows, two streams
  cudaStream_t stream[2] = {nullptr, nullptr};
  uint8_t* d_rows[2] = {nullptr, nullptr}; uint32_t* d_ff[2] = {nullptr, nullptr};
  size_t chunk = 0;
  std::mutex mu;
};

R1cs::~R1cs() {
  for (auto& kv : devs) {
    Dev* d = kv.second;
    int prev = -1;
    cudaGetDevice(&prev);
    cudaSetDevice(d->device);
    cudaFree(d->code); cudaFree(d->consts);
    for (int i = 0; i < 2; i++) { cudaFree(d->d_rows[i]); cudaFree(d->d_ff[i]); if (d->stream[i]) cudaStreamDestroy(d->stream[i]); }
    delete d;
    if (prev >= 0) cudaSetDevice(prev);
  }
}

// program and constant table, uploaded on first use of a device
R1cs::Dev* R1cs::dev(int device) {
  std::lock_guard<std::mutex> lk(mu);
  auto it = devs.find(device);
  if (it != devs.end()) return it->second;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) throw Error("no CUDA device available: this library has no CPU fallback");
  if (device < 0 || device >= ndev) throw Error("CUDA device index out of range");
  if (prog.code.size() / 2 > 0xFFFFFFFFull) throw Error("r1cs: program too large (more than 2^32 items)");
  DeviceGuard on(device);
  std::unique_ptr<Dev> d(new Dev());
  d->device = device;
  cudaDeviceProp prop; CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
  d->sms = prop.multiProcessorCount;
  d->smem_max = prop.sharedMemPerBlockOptin;
  CUDA_CHECK(cudaFuncSetAttribute(r1cs_check_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)d->smem_max));
  CUDA_CHECK(cudaMalloc(&d->code, std::max<size_t>(prog.code.size(), 2) * 4));
  CUDA_CHECK(cudaMemcpy(d->code, prog.code.data(), prog.code.size() * 4, cudaMemcpyHostToDevice));
  CUDA_CHECK(cudaMalloc(&d->consts, std::max<size_t>(prog.consts.size(), 1) * 32));
  CUDA_CHECK(cudaMemcpy(d->consts, prog.consts.data(), prog.consts.size() * 32, cudaMemcpyHostToDevice));
  devs[device] = d.get();
  return d.release();
}

void R1cs::check_device(int device, const void* d_witness, size_t B, size_t row_pitch, uint32_t* d_first_failed, void* stream) {
  const size_t row_b = (size_t)hdr.n_wires * 32;
  if (row_pitch < row_b) throw Error("row_pitch is smaller than n_wires x 32 bytes");
  if (row_pitch % 16 || ((uintptr_t)d_witness & 15)) throw Error("device witness rows must be 16-byte aligned (row_pitch a multiple of 16)");
  Dev* d = dev(device);
  if (B == 0) return;
  DeviceGuard on(device);
  cudaStream_t s = (cudaStream_t)stream;
  const uint32_t n_items = (uint32_t)(prog.code.size() / 2);
  if (n_items == 0) {                                   // no constraint: every row passes
    CUDA_CHECK(cudaMemsetAsync(d_first_failed, 0xFF, B * 4, s));
    return;
  }
  // threads per CTA: the smallest multiple of 32 that covers the batch with one wave of persistent CTAs, at most 512
  const size_t per_sm = (B + d->sms - 1) / d->sms;
  const int T = (int)std::min<size_t>(R1_MAX_THREADS, std::max<size_t>(32, (per_sm + 31) / 32 * 32));
  const size_t n_tiles = (B + T - 1) / T;
  if (n_tiles > 0xFFFFFFFFull) throw Error("batch too large");
  RParams p;
  p.code = d->code; p.n_items = n_items; p.consts = d->consts;
  p.witness = (const uint8_t*)d_witness; p.pitch = row_pitch; p.B = B;
  p.n_constraints = hdr.n_constraints; p.n_tiles = (uint32_t)n_tiles; p.first_failed = d_first_failed;
  const size_t ring_b = (size_t)(T / 32) * R1_RING * 8;
  p.n_hot = (uint32_t)std::min<size_t>(prog.consts.size(), (d->smem_max - ring_b) / 32);
  const int grid = (int)std::min<size_t>(n_tiles, (size_t)d->sms);
  r1cs_check_kernel<<<grid, T, (size_t)p.n_hot * 32 + ring_b, s>>>(p);
  CUDA_CHECK(cudaGetLastError());
}

namespace {
// no copy may still target the caller's memory when a host-buffer call returns, also on errors
struct Drain {
  cudaStream_t a, b;
  ~Drain() { if (a) cudaStreamSynchronize(a); if (b) cudaStreamSynchronize(b); }
};
}  // namespace

// host rows: chunked, double-buffered H2D (pitched) -> check -> D2H of the verdicts on two streams
void R1cs::check_host_on(int device, const uint8_t* witness, size_t B, size_t row_pitch, uint32_t* first_failed) {
  Dev* d = dev(device);
  DeviceGuard on(device);
  std::lock_guard<std::mutex> lk(d->mu);
  const size_t row_b = (size_t)hdr.n_wires * 32, dev_row = std::max<size_t>(row_b, 16);
  size_t free_b = 0, total_b = 0;
  CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
  // two staging buffers of at most 8 GiB each, and together at most 2/5 of what is free
  const size_t budget = std::min<size_t>((size_t)8 << 30, (free_b + 2 * d->chunk * (dev_row + 4)) / 5);
  size_t chunk = std::max<size_t>(1, budget / (dev_row + 4));
  if (B >= 4 * 1024) chunk = std::min(chunk, (B + 3) / 4);        // at least four chunks: copies overlap the checks
  chunk = std::min(chunk, B);
  if (chunk > d->chunk) {
    d->chunk = 0;
    for (int i = 0; i < 2; i++) { cudaFree(d->d_rows[i]); d->d_rows[i] = nullptr; cudaFree(d->d_ff[i]); d->d_ff[i] = nullptr; }
    for (int i = 0; i < 2; i++) {
      CUDA_CHECK(cudaMalloc(&d->d_rows[i], chunk * dev_row));
      CUDA_CHECK(cudaMalloc(&d->d_ff[i], chunk * 4));
      if (!d->stream[i]) CUDA_CHECK(cudaStreamCreateWithFlags(&d->stream[i], cudaStreamNonBlocking));
    }
    d->chunk = chunk;
  }
  Drain drain{d->stream[0], d->stream[1]};
  int k = 0;
  for (size_t off = 0; off < B; off += chunk, k ^= 1) {
    const size_t nb = std::min(chunk, B - off);
    cudaStream_t s = d->stream[k];
    if (row_b == 0) {}
    else if (row_pitch == row_b) CUDA_CHECK(cudaMemcpyAsync(d->d_rows[k], witness + off * row_pitch, nb * row_b, cudaMemcpyHostToDevice, s));
    else CUDA_CHECK(cudaMemcpy2DAsync(d->d_rows[k], dev_row, witness + off * row_pitch, row_pitch, row_b, nb, cudaMemcpyHostToDevice, s));
    check_device(device, d->d_rows[k], nb, dev_row, d->d_ff[k], s);
    CUDA_CHECK(cudaMemcpyAsync(first_failed + off, d->d_ff[k], nb * 4, cudaMemcpyDeviceToHost, s));
  }
  CUDA_CHECK(cudaStreamSynchronize(d->stream[0]));
  CUDA_CHECK(cudaStreamSynchronize(d->stream[1]));
}

void R1cs::check_host(const uint8_t* witness, size_t B, size_t row_pitch, uint32_t* first_failed, int n_gpus, int first_device) {
  if (row_pitch < (size_t)hdr.n_wires * 32) throw Error("row_pitch is smaller than n_wires x 32 bytes");
  if (B == 0) return;
  if (n_gpus <= 1) { check_host_on(first_device, witness, B, row_pitch, first_failed); return; }
  // independent rows: contiguous shards, one host thread per GPU, no collective
  std::vector<std::thread> th;
  std::vector<std::string> errs(n_gpus);
  for (int g = 0; g < n_gpus; g++) {
    const size_t lo = B * g / n_gpus, hi = B * (g + 1) / n_gpus;
    if (hi == lo) continue;
    th.emplace_back([=, &errs]() {
      try {
        bind_thread_near_device(first_device + g);
        check_host_on(first_device + g, witness + lo * row_pitch, hi - lo, row_pitch, first_failed + lo);
      } catch (const std::exception& e) { errs[g] = e.what(); }
    });
  }
  for (auto& t : th) t.join();
  for (auto& e : errs) if (!e.empty()) throw Error(e);
}

}  // namespace gw
