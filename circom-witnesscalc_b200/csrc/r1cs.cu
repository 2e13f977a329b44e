// R1CS check of witness rows on sm_100a: for every row, the lowest constraint k with <A_k,w> * <B_k,w> != <C_k,w>.
//
// Execution model: one thread = one witness row, so the 32 lanes of a warp check 32 rows against the SAME constraint
// stream (warp-uniform control flow, no divergence).  Each warp streams the 8-byte program items itself, as
// eval_batch_kernel streams its instruction slots: lane l loads item base + l (one coalesced 256-byte read), two
// blocks of 32 are staged in the warp's ring in shared memory, the next block waits in a register, and every lane
// reads the current item from shared memory (a broadcast).  The most used constants are staged in shared memory
// once per CTA.  A term reads the 32 bytes of its wire from the lane's own row: two 16-byte loads of one sector.
// Persistent CTAs (one per SM) walk tiles of rows; a warp whose 32 rows have all failed stops early.
// r1cs_abc_kernel runs the same stream, term loop and launch shape to store <A_k,w>, <B_k,w>, <C_k,w> of every row.
#include <cuda_runtime.h>

#include <algorithm>
#include <memory>
#include <string>
#include <vector>

#include "cuda_util.hpp"
#include "ntt.hpp"
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

// the ABC evaluation: the check's parameters (first_failed may be NULL: no verdict) and the output rows
struct AParams {
  RParams r;
  uint8_t* abc; unsigned long long abc_pitch;
  uint32_t n;                            // entries per vector; entries n_constraints .. n - 1 are the Groth16 tail
  uint32_t n_pub;                        // tail entry n_constraints + s, s <= n_pub, has A = w_s
};

const int R1_RING = 64;                  // program items staged per warp (two blocks of 32)
const int R1_MAX_THREADS = 512;          // one persistent CTA per SM; 512 threads x 128 registers = the register file

}  // namespace

// 32 bytes at v (two 16-byte loads of one sector) as a field element
__device__ __forceinline__ fe r1cs_load(const uint4* v) {
  fe r;
  const uint4 lo = __ldg(v), hi = __ldg(v + 1);
  r.l[0] = lo.x; r.l[1] = lo.y; r.l[2] = lo.z; r.l[3] = lo.w; r.l[4] = hi.x; r.l[5] = hi.y; r.l[6] = hi.z; r.l[7] = hi.w;
  return r;
}

// table constant c: from shared memory when it is one of the n_hot staged ones
__device__ __forceinline__ fe r1cs_const(const uint4* hot, const RParams& p, uint32_t c) {
  fe r;
  const uint4 lo = c < p.n_hot ? hot[2 * c] : __ldg(p.consts + 2 * (size_t)c);
  const uint4 hi = c < p.n_hot ? hot[2 * c + 1] : __ldg(p.consts + 2 * (size_t)c + 1);
  r.l[0] = lo.x; r.l[1] = lo.y; r.l[2] = lo.z; r.l[3] = lo.w; r.l[4] = hi.x; r.l[5] = hi.y; r.l[6] = hi.z; r.l[7] = hi.w;
  return r;
}

// The warp's constraint stream from item 0: blocks 0 and 1 staged in the ring, block 2 in flight in nblk.
// next(a, b) yields the next item.
struct ProgramStream {
  uint2* ring; const uint2* code; uint32_t n; uint32_t lane; uint32_t pc; uint2 nblk;
  __device__ __forceinline__ ProgramStream(uint2* ring_, const uint2* code_, uint32_t n_, uint32_t lane_)
      : ring(ring_), code(code_), n(n_), lane(lane_), pc(0) {
    __syncwarp();
    ring[lane] = __ldg(code + min(lane, n - 1));
    ring[32 + lane] = __ldg(code + min(32u + lane, n - 1));
    nblk = __ldg(code + min(64u + lane, n - 1));
    __syncwarp();
  }
  __device__ __forceinline__ void operator()(uint32_t& a, uint32_t& b) {
    const uint2 it = ring[pc & (R1_RING - 1)];
    a = it.x; b = it.y;
    pc++;
    if ((pc & 31u) == 0) {
      // block (pc >> 5) - 1 is consumed: stage block (pc >> 5) + 1 in its half, start loading the one after it
      __syncwarp();
      ring[(((pc >> 5) - 1) & 1u) * 32u + lane] = nblk;
      nblk = __ldg(code + min(((pc >> 5) + 2u) * 32u + lane, n - 1));
      __syncwarp();
    }
  }
};

// Dynamic shared memory: [n_hot][2] hot constants (uint4) | [T/32 warps][R1_RING] program items (uint2).
__global__ void __launch_bounds__(R1_MAX_THREADS, 1) r1cs_check_kernel(const RParams p) {
  extern __shared__ uint4 smem[];
  const int T = blockDim.x;
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const uint4* hot = smem;
  uint2* ring = reinterpret_cast<uint2*>(smem + 2 * (size_t)p.n_hot) + (tid >> 5) * R1_RING;

  for (uint32_t k = tid; k < 2 * p.n_hot; k += T) smem[k] = __ldg(p.consts + k);
  __syncthreads();

  auto const_val = [&](uint32_t c) { return r1cs_const(hot, p, c); };

  for (uint32_t tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
    const unsigned long long row = (unsigned long long)tile * T + tid;
    const bool active = row < p.B;
    if (__all_sync(0xFFFFFFFFu, !active)) continue;
    const uint4* w = reinterpret_cast<const uint4*>(p.witness + (active ? row : p.B - 1) * p.pitch);
    auto wire_val = [&](uint32_t i) { return r1cs_load(w + 2 * (size_t)i); };
    ProgramStream next(ring, p.code, p.n_items, lane);

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

// A, B and C of every constraint for every row, in the layout of gw_r1cs_abc_batch: the check kernel's stream, term loop
// and launch shape, with wire values reduced mod M (r1cs_wire_reduce), no early exit, and the values stored as soon as
// they are reduced: two 16-byte streaming stores, one 32-byte sector, to the lane's own output row.  The Groth16 tail
// (public-input rows, then zeros) follows on the same lane.  VERDICT: the check's first_failed, bit for bit; without
// it no product a * b is computed.
template <bool VERDICT>
__global__ void __launch_bounds__(R1_MAX_THREADS, 1) r1cs_abc_kernel(const AParams q) {
  const RParams& p = q.r;
  extern __shared__ uint4 smem[];
  const int T = blockDim.x;
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const uint4* hot = smem;
  uint2* ring = reinterpret_cast<uint2*>(smem + 2 * (size_t)p.n_hot) + (tid >> 5) * R1_RING;

  for (uint32_t k = tid; k < 2 * p.n_hot; k += T) smem[k] = __ldg(p.consts + k);
  __syncthreads();

  auto const_val = [&](uint32_t c) { return r1cs_const(hot, p, c); };
  const size_t vec = 2 * (size_t)q.n;          // uint4 per vector

  for (uint32_t tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
    const unsigned long long row = (unsigned long long)tile * T + tid;
    const bool active = row < p.B;
    if (__all_sync(0xFFFFFFFFu, !active)) continue;
    const uint4* w = reinterpret_cast<const uint4*>(p.witness + (active ? row : p.B - 1) * p.pitch);
    uint4* out = reinterpret_cast<uint4*>(q.abc + (active ? row : 0) * q.abc_pitch);
    auto wire_val = [&](uint32_t i) { return r1cs_load(w + 2 * (size_t)i); };
    auto store = [&](size_t at, const fe& v) {
      if (active) {
        __stcs(out + at, make_uint4(v.l[0], v.l[1], v.l[2], v.l[3]));
        __stcs(out + at + 1, make_uint4(v.l[4], v.l[5], v.l[6], v.l[7]));
      }
    };
    ProgramStream next(ring, p.code, p.n_items, lane);

    uint32_t first = R1CS_OK;
#pragma unroll 1
    for (uint32_t k = 0; k < p.n_constraints; k++) {
      bool reduced = false;
      fe a, b;
      r1cs_abc(next, wire_val, const_val, &reduced, [&](int which, const fe& v) {
        store(which * vec + 2 * (size_t)k, v);
        if (VERDICT) {
          if (which == 0) a = v;
          else if (which == 1) b = v;
          else if (first == R1CS_OK && (reduced || !r1cs_holds(a, b, v))) first = k;
        }
      });
    }
#pragma unroll 1
    for (uint32_t j = p.n_constraints; j < q.n; j++) {
      const uint32_t s = j - p.n_constraints;
      bool unused = false;
      store(2 * (size_t)j, s <= q.n_pub ? r1cs_wire_reduce(wire_val(s), &unused) : fe_zero());
      store(vec + 2 * (size_t)j, fe_zero());
      store(2 * vec + 2 * (size_t)j, fe_zero());
    }
    if (VERDICT && active) p.first_failed[row] = first;
  }
}

struct R1cs::Dev {
  int device = -1;
  int sms = 0;
  size_t smem_max = 0;
  uint2* code = nullptr; uint4* consts = nullptr;
  // staging of the host-row entry points: two chunks of dense rows (and of their results), two streams
  cudaStream_t stream[2] = {nullptr, nullptr};
  uint8_t* d_rows[2] = {nullptr, nullptr}; uint32_t* d_ff[2] = {nullptr, nullptr}; uint8_t* d_out[2] = {nullptr, nullptr};
  size_t chunk = 0, out_b = 0;             // rows per chunk; bytes of each d_out
  std::mutex mu;
  ~Dev() {
    int prev = -1;
    cudaGetDevice(&prev);
    cudaSetDevice(device);
    cudaFree(code); cudaFree(consts);
    for (int i = 0; i < 2; i++) {
      cudaFree(d_rows[i]); cudaFree(d_ff[i]); cudaFree(d_out[i]);
      if (stream[i]) cudaStreamDestroy(stream[i]);
    }
    if (prev >= 0) cudaSetDevice(prev);
  }
};

R1cs::R1cs(const uint8_t* data, size_t len) { parse_r1cs(data, len, hdr, prog); }
R1cs::~R1cs() = default;

// program and constant table, uploaded on first use of a device
R1cs::Dev* R1cs::dev(int device) {
  std::lock_guard<std::mutex> lk(mu);
  auto it = devs.find(device);
  if (it != devs.end()) return it->second.get();
  gw::check_device(device);   // the free function, not R1cs::check_device
  if (prog.code.size() / 2 > 0xFFFFFFFFull) throw Error("r1cs: program too large (more than 2^32 items)");
  DeviceGuard on(device);
  std::unique_ptr<Dev> d(new Dev());
  d->device = device;
  cudaDeviceProp prop; CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
  d->sms = prop.multiProcessorCount;
  d->smem_max = prop.sharedMemPerBlockOptin;
  CUDA_CHECK(cudaFuncSetAttribute(r1cs_check_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)d->smem_max));
  CUDA_CHECK(cudaFuncSetAttribute(r1cs_abc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)d->smem_max));
  CUDA_CHECK(cudaFuncSetAttribute(r1cs_abc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)d->smem_max));
  CUDA_CHECK(cudaMalloc(&d->code, std::max<size_t>(prog.code.size(), 2) * 4));
  CUDA_CHECK(cudaMemcpy(d->code, prog.code.data(), prog.code.size() * 4, cudaMemcpyHostToDevice));
  CUDA_CHECK(cudaMalloc(&d->consts, std::max<size_t>(prog.consts.size(), 1) * 32));
  CUDA_CHECK(cudaMemcpy(d->consts, prog.consts.data(), prog.consts.size() * 32, cudaMemcpyHostToDevice));
  return (devs[device] = std::move(d)).get();
}

struct R1cs::Launch {
  RParams p;
  int grid, threads;
  size_t smem;
};

// kernel parameters and launch shape of B rows: persistent CTAs, one per SM; threads per CTA the smallest multiple of 32
// that covers the batch with one wave, at most 512
R1cs::Launch R1cs::launch(Dev* d, const void* d_witness, size_t B, size_t row_pitch, uint32_t* d_first_failed) const {
  const size_t per_sm = (B + d->sms - 1) / d->sms;
  const int T = (int)std::min<size_t>(R1_MAX_THREADS, std::max<size_t>(32, (per_sm + 31) / 32 * 32));
  const size_t n_tiles = (B + T - 1) / T;
  if (n_tiles > 0xFFFFFFFFull) throw Error("batch too large");
  Launch l;
  RParams& p = l.p;
  p.code = d->code; p.n_items = (uint32_t)(prog.code.size() / 2); p.consts = d->consts;
  p.witness = (const uint8_t*)d_witness; p.pitch = row_pitch; p.B = B;
  p.n_constraints = hdr.n_constraints; p.n_tiles = (uint32_t)n_tiles; p.first_failed = d_first_failed;
  const size_t ring_b = (size_t)(T / 32) * R1_RING * 8;
  p.n_hot = (uint32_t)std::min<size_t>(prog.consts.size(), (d->smem_max - ring_b) / 32);
  l.grid = (int)std::min<size_t>(n_tiles, (size_t)d->sms);
  l.threads = T;
  l.smem = (size_t)p.n_hot * 32 + ring_b;
  return l;
}

void R1cs::check_device(int device, const void* d_witness, size_t B, size_t row_pitch, uint32_t* d_first_failed, void* stream) {
  const size_t row_b = (size_t)hdr.n_wires * 32;
  if (row_pitch < row_b) throw Error("row_pitch is smaller than n_wires x 32 bytes");
  if (row_pitch % 16 || ((uintptr_t)d_witness & 15)) throw Error("device witness rows must be 16-byte aligned (row_pitch a multiple of 16)");
  Dev* d = dev(device);
  if (B == 0) return;
  DeviceGuard on(device);
  cudaStream_t s = (cudaStream_t)stream;
  if (prog.code.empty()) {                              // no constraint: every row passes
    CUDA_CHECK(cudaMemsetAsync(d_first_failed, 0xFF, B * 4, s));
    return;
  }
  const Launch l = launch(d, d_witness, B, row_pitch, d_first_failed);
  r1cs_check_kernel<<<l.grid, l.threads, l.smem, s>>>(l.p);
  CUDA_CHECK(cudaGetLastError());
}

uint64_t R1cs::abc_len(uint32_t options) const {
  if (options & ~R1CS_ABC_GROTH16) throw Error("unknown option bits " + std::to_string(options & ~R1CS_ABC_GROTH16) + " (known: GW_R1CS_ABC_GROTH16)");
  if (!(options & R1CS_ABC_GROTH16)) return hdr.n_constraints;
  const uint64_t n_pub = (uint64_t)hdr.n_pub_out + hdr.n_pub_in;
  if (n_pub >= hdr.n_wires)
    throw Error("r1cs: " + std::to_string(n_pub) + " public signals need more than the " + std::to_string(hdr.n_wires) + " wires");
  uint64_t n = 1;
  while (n < hdr.n_constraints + n_pub + 1) n <<= 1;
  if (n > (1ull << 31)) throw Error("r1cs: the Groth16 domain is larger than 2^31");
  return n;
}

size_t R1cs::abc_row_bytes(size_t row_pitch, size_t abc_pitch, uint32_t options, bool device) const {
  const size_t out_b = 3 * 32 * (size_t)abc_len(options);
  if (row_pitch < (size_t)hdr.n_wires * 32) throw Error("row_pitch is smaller than n_wires x 32 bytes");
  if (abc_pitch < out_b) throw Error("abc_pitch is smaller than 3 x n x 32 bytes (n = gw_r1cs_abc_len)");
  if (device && (row_pitch % 16 || abc_pitch % 16)) throw Error("device rows must be 16-byte aligned (row_pitch and abc_pitch multiples of 16)");
  return out_b;
}

void R1cs::abc_device(int device, const void* d_witness, size_t B, size_t row_pitch, void* d_abc, size_t abc_pitch,
                      uint32_t options, uint32_t* d_first_failed, void* stream) {
  abc_row_bytes(row_pitch, abc_pitch, options, true);
  if (((uintptr_t)d_witness & 15) || ((uintptr_t)d_abc & 15)) throw Error("device buffers must be 16-byte aligned");
  if (B == 0) return;
  Dev* d = dev(device);
  DeviceGuard on(device);
  AParams q;
  q.n = (uint32_t)abc_len(options);
  q.n_pub = hdr.n_pub_out + hdr.n_pub_in;
  q.abc = (uint8_t*)d_abc; q.abc_pitch = abc_pitch;
  const Launch l = launch(d, d_witness, B, row_pitch, d_first_failed);
  q.r = l.p;
  // without constraints the stream's prefetch still reads item 0 (the allocation holds at least one); none is consumed
  q.r.n_items = std::max<uint32_t>(q.r.n_items, 1);
  if (d_first_failed) r1cs_abc_kernel<true><<<l.grid, l.threads, l.smem, (cudaStream_t)stream>>>(q);
  else r1cs_abc_kernel<false><<<l.grid, l.threads, l.smem, (cudaStream_t)stream>>>(q);
  CUDA_CHECK(cudaGetLastError());
}

// host rows: chunked, double-buffered H2D (pitched) -> check, ABC or quotient -> D2H of the results on two streams.
// out == NULL: the check; else the ABC vectors or h (and the verdicts when first_failed is not NULL).  The chunk size
// counts the 3 x n x 32 device bytes of a row in both output modes; only h (n x 32 bytes) of a quotient row is copied.
void R1cs::host_rows_on(int device, const uint8_t* witness, size_t B, size_t row_pitch, uint32_t* first_failed, const AbcOut* out) {
  Dev* d = dev(device);
  DeviceGuard on(device);
  std::lock_guard<std::mutex> lk(d->mu);
  const size_t row_b = (size_t)hdr.n_wires * 32, dev_row = std::max<size_t>(row_b, 16);
  const size_t out_row = out ? 3 * 32 * (size_t)abc_len(out->options) : 0;
  const size_t copy_b = out && out->quotient ? out_row / 3 : out_row;       // bytes of a result row copied back
  size_t free_b = 0, total_b = 0;
  CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
  // two staging buffers of at most 8 GiB each, and together at most 2/5 of what is free
  const size_t budget = std::min<size_t>((size_t)8 << 30, (free_b + 2 * (d->chunk * (dev_row + 4) + d->out_b)) / 5);
  size_t chunk = std::max<size_t>(1, budget / (dev_row + 4 + out_row));
  if (B >= 4 * 1024) chunk = std::min(chunk, (B + 3) / 4);        // at least four chunks: copies overlap the kernels
  chunk = std::min(chunk, B);
  if (chunk > d->chunk || chunk * out_row > d->out_b) {
    d->chunk = 0; d->out_b = 0;
    for (int i = 0; i < 2; i++) {
      cudaFree(d->d_rows[i]); d->d_rows[i] = nullptr; cudaFree(d->d_ff[i]); d->d_ff[i] = nullptr;
      cudaFree(d->d_out[i]); d->d_out[i] = nullptr;
    }
    for (int i = 0; i < 2; i++) {
      CUDA_CHECK(cudaMalloc(&d->d_rows[i], chunk * dev_row));
      CUDA_CHECK(cudaMalloc(&d->d_ff[i], chunk * 4));
      if (out_row) CUDA_CHECK(cudaMalloc(&d->d_out[i], chunk * out_row));
      if (!d->stream[i]) CUDA_CHECK(cudaStreamCreateWithFlags(&d->stream[i], cudaStreamNonBlocking));
    }
    d->chunk = chunk; d->out_b = chunk * out_row;
  }
  StreamDrain drain{d->stream[0], d->stream[1]};
  int k = 0;
  for (size_t off = 0; off < B; off += chunk, k ^= 1) {
    const size_t nb = std::min(chunk, B - off);
    cudaStream_t s = d->stream[k];
    if (row_b == 0) {}
    else if (row_pitch == row_b) CUDA_CHECK(cudaMemcpyAsync(d->d_rows[k], witness + off * row_pitch, nb * row_b, cudaMemcpyHostToDevice, s));
    else CUDA_CHECK(cudaMemcpy2DAsync(d->d_rows[k], dev_row, witness + off * row_pitch, row_pitch, row_b, nb, cudaMemcpyHostToDevice, s));
    if (!out) check_device(device, d->d_rows[k], nb, dev_row, d->d_ff[k], s);
    else {
      if (out->quotient) quotient_device(device, d->d_rows[k], nb, dev_row, d->d_out[k], out_row, first_failed ? d->d_ff[k] : nullptr, s);
      else abc_device(device, d->d_rows[k], nb, dev_row, d->d_out[k], out_row, out->options, first_failed ? d->d_ff[k] : nullptr, s);
      if (out_row == 0) {}
      else if (out->pitch == out_row && copy_b == out_row) CUDA_CHECK(cudaMemcpyAsync(out->abc + off * out_row, d->d_out[k], nb * out_row, cudaMemcpyDeviceToHost, s));
      else CUDA_CHECK(cudaMemcpy2DAsync(out->abc + off * out->pitch, out->pitch, d->d_out[k], out_row, copy_b, nb, cudaMemcpyDeviceToHost, s));
    }
    if (first_failed) CUDA_CHECK(cudaMemcpyAsync(first_failed + off, d->d_ff[k], nb * 4, cudaMemcpyDeviceToHost, s));
  }
  CUDA_CHECK(cudaStreamSynchronize(d->stream[0]));
  CUDA_CHECK(cudaStreamSynchronize(d->stream[1]));
}

void R1cs::host_rows(const uint8_t* witness, size_t B, size_t row_pitch, uint32_t* first_failed, const AbcOut* out, int n_gpus,
                     int first_device) {
  if (B == 0) return;
  if (n_gpus <= 1) { host_rows_on(first_device, witness, B, row_pitch, first_failed, out); return; }
  run_shards(B, n_gpus, first_device, [&](int device, size_t lo, size_t hi) {
    AbcOut shard;
    if (out) shard = AbcOut{out->abc + lo * out->pitch, out->pitch, out->options, out->quotient};
    host_rows_on(device, witness + lo * row_pitch, hi - lo, row_pitch, first_failed ? first_failed + lo : nullptr, out ? &shard : nullptr);
  });
}

void R1cs::check_host(const uint8_t* witness, size_t B, size_t row_pitch, uint32_t* first_failed, int n_gpus, int first_device) {
  if (row_pitch < (size_t)hdr.n_wires * 32) throw Error("row_pitch is smaller than n_wires x 32 bytes");
  host_rows(witness, B, row_pitch, first_failed, nullptr, n_gpus, first_device);
}

void R1cs::abc_host(const uint8_t* witness, size_t B, size_t row_pitch, uint8_t* abc, size_t abc_pitch, uint32_t options,
                    uint32_t* first_failed, int n_gpus, int first_device) {
  abc_row_bytes(row_pitch, abc_pitch, options, false);
  const AbcOut out{abc, abc_pitch, options, false};
  host_rows(witness, B, row_pitch, first_failed, &out, n_gpus, first_device);
}

uint32_t R1cs::quotient_log_n(size_t row_pitch, size_t out_pitch, bool device) const {
  const uint64_t n = abc_len(R1CS_ABC_GROTH16);
  uint32_t log_n = 0;
  while ((1ull << log_n) < n) log_n++;
  if (log_n > NTT_MAX_LOG)
    throw Error("r1cs: the Groth16 domain 2^" + std::to_string(log_n) + " is larger than 2^24: domains above 2^24 are not supported");
  if (row_pitch < (size_t)hdr.n_wires * 32) throw Error("row_pitch is smaller than n_wires x 32 bytes");
  if (device && out_pitch < 3 * 32 * n) throw Error("work_pitch is smaller than 3 x n x 32 bytes (n = gw_r1cs_abc_len)");
  if (!device && out_pitch < 32 * n) throw Error("h_pitch is smaller than n x 32 bytes (n = gw_r1cs_abc_len)");
  if (device && (row_pitch % 16 || out_pitch % 16)) throw Error("device rows must be 16-byte aligned (row_pitch and work_pitch multiples of 16)");
  return log_n;
}

void R1cs::quotient_device(int device, const void* d_witness, size_t B, size_t row_pitch, void* d_work, size_t work_pitch,
                           uint32_t* d_first_failed, void* stream) {
  const uint32_t log_n = quotient_log_n(row_pitch, work_pitch, true);
  if (((uintptr_t)d_witness & 15) || ((uintptr_t)d_work & 15)) throw Error("device buffers must be 16-byte aligned");
  if (B == 0) return;
  abc_device(device, d_witness, B, row_pitch, d_work, work_pitch, R1CS_ABC_GROTH16, d_first_failed, stream);
  ntt_quotient_device(device, d_work, B, log_n, work_pitch, stream);
}

void R1cs::quotient_host(const uint8_t* witness, size_t B, size_t row_pitch, uint8_t* h, size_t h_pitch, uint32_t* first_failed,
                         int n_gpus, int first_device) {
  quotient_log_n(row_pitch, h_pitch, false);
  const AbcOut out{h, h_pitch, R1CS_ABC_GROTH16, true};
  host_rows(witness, B, row_pitch, first_failed, &out, n_gpus, first_device);
}

}  // namespace gw
