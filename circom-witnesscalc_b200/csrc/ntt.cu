// Batched BN254 NTTs on sm_100a (gw_fr_ntt_batch_device) and the Groth16 quotient transforms of ABC rows.
//
// A CTA transforms whole sub-vectors in shared memory with radix-2 stages (ntt_smem): one butterfly per thread and
// stage, twiddles from the w_4096 table (__ldg), one __syncthreads per stage.  Every multiplication is ntt_mul
// (ntt.cuh): dot_mac + one Montgomery reduction against a pre-scaled twiddle.
//   n <= 2^12: the whole vector in one CTA (ntt_small_kernel, ntt_small_quotient_kernel).
//   n = n1 * n2 > 2^12 (n2 = 2^floor(k/2) <= n1 <= 2^12): the four-step split, in place.  Index i = i1 + n1 i2.
//     column pass (ntt_col_kernel): for each i1, the n2 entries i1 + n1 i2 (stride n1), DIF -> bit-reversed slot p,
//       times w_n^(i1 rev(p)), back to i1 + n1 p.  A CTA takes C adjacent columns, so C lanes read C * 32 contiguous
//       bytes of each row.
//     row pass (ntt_row_kernel): each block of n1 contiguous entries, DIF.  Entry P then holds y[rev_n(P)].
//   Natural order out of the standalone transform needs the permutation rev_n: ntt_bitrev_kernel swaps 16 x 16 tiles
//   (runs of 16 contiguous entries, 512 bytes).  The quotient never permutes: its inverse is this DIF, its forward the
//   transposed algorithm (DIT, bit-reversed in, natural out), which starts on the same row blocks, so the row pass does
//   inverse DIF, the coset factor n^-1 g^i and forward DIT in one shared-memory visit, and the last column pass (DIT)
//   reads A, B and C of a column and writes h = A B - C once.
// Coset factors and n^-1 are fused into the first or last pass; twiddle tables are built once per (device, k).
#include <cuda_runtime.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <string>
#include <utility>

#include "cuda_util.hpp"
#include "ntt.cuh"

namespace gw {

namespace {

const int NTT_THREADS = 256;
const uint32_t NTT_CTA_ELEMS = 2048;       // entries a CTA aims to hold (64 KB: two CTAs per SM); a 4096-entry
                                           // sub-transform takes 128 KB

struct NttArgs {
  uint8_t* base; unsigned long long pitch, vec_b;   // vector v at base + (v / per_row) * pitch + (v % per_row) * vec_b
  uint32_t per_row;
  unsigned long long n_vectors;                     // vectors (standalone) or rows (quotient)
  uint32_t lg, lg1, lg2;                            // n = 2^lg = n1 * n2
  uint32_t C;                                       // sub-transforms per CTA
  uint32_t flags;
  const uint4* tab;                                 // ntt_build_tables(lg)
};

__device__ __forceinline__ fe ld_s(const uint4* p) {
  const uint4 lo = p[0], hi = p[1];
  fe r;
  r.l[0] = lo.x; r.l[1] = lo.y; r.l[2] = lo.z; r.l[3] = lo.w; r.l[4] = hi.x; r.l[5] = hi.y; r.l[6] = hi.z; r.l[7] = hi.w;
  return r;
}
__device__ __forceinline__ fe ld_tab(const uint4* tab, uint32_t j, uint32_t t) {
  const uint4* p = tab + 2 * ((size_t)j * NTT_TAB + t);
  const uint4 lo = __ldg(p), hi = __ldg(p + 1);
  fe r;
  r.l[0] = lo.x; r.l[1] = lo.y; r.l[2] = lo.z; r.l[3] = lo.w; r.l[4] = hi.x; r.l[5] = hi.y; r.l[6] = hi.z; r.l[7] = hi.w;
  return r;
}
__device__ __forceinline__ void st_s(uint4* p, const fe& v) {
  p[0] = make_uint4(v.l[0], v.l[1], v.l[2], v.l[3]);
  p[1] = make_uint4(v.l[4], v.l[5], v.l[6], v.l[7]);
}
__device__ __forceinline__ uint4* vec_ptr(const NttArgs& a, unsigned long long v) {
  return reinterpret_cast<uint4*>(a.base + (v / a.per_row) * a.pitch + (v % a.per_row) * a.vec_b);
}
__device__ __forceinline__ uint32_t rev(uint32_t x, uint32_t lg) { return lg ? __brev(x) >> (32 - lg) : 0u; }
__device__ __forceinline__ fe reduce_in(fe x) {
  if (x.l[7] >= MOD_L(7) && fe_geq_m(x)) x = fe_reduce256(x);
  return x;
}
// x * r^e (e < 2^24) for the power tables LO, HI of one root: HI[0] = 1, so e < 4096 takes one multiplication
__device__ __forceinline__ fe mul_pow(const fe& x, const uint4* tab, uint32_t lo, uint32_t hi, uint32_t e) {
  fe r = ntt_mul(x, ld_tab(tab, lo, e & (NTT_TAB - 1)));
  if (e >> 12) r = ntt_mul(r, ld_tab(tab, hi, e >> 12));
  return r;
}

// C transforms of 2^lg entries in shared memory, transform c at entry c * stride.  DIF: natural in, bit-reversed out;
// else DIT: bit-reversed in, natural out.  root: the w_4096 powers of the direction.  Ends with __syncthreads.
template <bool DIF>
__device__ __forceinline__ void ntt_smem(uint4* s, uint32_t C, uint32_t lg, uint32_t stride, const uint4* tab, uint32_t root) {
  if (lg == 0) return;
  const uint32_t nb = C << (lg - 1), hmask = (1u << (lg - 1)) - 1;
#pragma unroll 1
  for (uint32_t stage = 0; stage < lg; stage++) {
    const uint32_t lgh = DIF ? lg - 1 - stage : stage;
    const uint32_t h = 1u << lgh;
#pragma unroll 1
    for (uint32_t t = threadIdx.x; t < nb; t += blockDim.x) {
      const uint32_t c = t >> (lg - 1), u = t & hmask, j = u & (h - 1);
      uint4* p = s + 2 * (c * stride + ((u >> lgh) << (lgh + 1)) + j);
      fe x = ld_s(p), y = ld_s(p + 2 * h);
      const fe w = ld_tab(tab, root, j << (11 - lgh));      // w_2h^j = w_4096^(j 2048 / h)
      if (DIF) ntt_bfly_dif(x, y, w); else ntt_bfly_dit(x, y, w);
      st_s(p, x);
      st_s(p + 2 * h, y);
    }
    __syncthreads();
  }
}

}  // namespace

// n <= 2^12: C whole vectors per CTA, natural order in and out (the permutation is a shared-memory read).
__global__ void __launch_bounds__(NTT_THREADS, 2) ntt_small_kernel(const NttArgs a) {
  extern __shared__ uint4 sm[];
  const uint32_t n = 1u << a.lg;
  const unsigned long long v0 = (unsigned long long)blockIdx.x * a.C;
  const uint32_t nv = (uint32_t)min((unsigned long long)a.C, a.n_vectors - v0);
  const bool inv = a.flags & NTT_INVERSE, coset = a.flags & NTT_COSET;
#pragma unroll 1
  for (uint32_t e = threadIdx.x; e < (nv << a.lg); e += blockDim.x) {
    const uint32_t i = e & (n - 1);
    fe x = reduce_in(ld_s(vec_ptr(a, v0 + (e >> a.lg)) + 2 * i));
    if (coset && !inv) x = ntt_mul(x, ld_tab(a.tab, CG_LO, i));
    st_s(sm + 2 * e, x);
  }
  __syncthreads();
  ntt_smem<true>(sm, nv, a.lg, n, a.tab, inv ? IROOT : ROOT);
#pragma unroll 1
  for (uint32_t e = threadIdx.x; e < (nv << a.lg); e += blockDim.x) {
    const uint32_t v = e >> a.lg, j = e & (n - 1);
    fe y = ld_s(sm + 2 * ((v << a.lg) + rev(j, a.lg)));
    if (inv) y = ntt_mul(y, coset ? ld_tab(a.tab, ICG_LO, j) : ld_tab(a.tab, NINV, 0));
    st_s(vec_ptr(a, v0 + v) + 2 * j, y);
  }
}

// The quotient of one row per CTA, n <= 2^12: for X = A, B, C the inverse DIF, n^-1 g^i, the forward DIT, then
// A_odd (pre-scaled) is stored in the A slot, A_odd B_odd replaces it, and h = A_odd B_odd - C_odd replaces that.
__global__ void __launch_bounds__(NTT_THREADS, 2) ntt_small_quotient_kernel(const NttArgs a) {
  extern __shared__ uint4 sm[];
  const uint32_t n = 1u << a.lg;
  uint4* row = reinterpret_cast<uint4*>(a.base + (unsigned long long)blockIdx.x * a.pitch);
#pragma unroll 1
  for (uint32_t which = 0; which < 3; which++) {
    const uint4* x = row + 2 * (size_t)which * n;
#pragma unroll 1
    for (uint32_t e = threadIdx.x; e < n; e += blockDim.x) st_s(sm + 2 * e, ld_s(x + 2 * e));
    __syncthreads();
    ntt_smem<true>(sm, 1, a.lg, n, a.tab, IROOT);
#pragma unroll 1
    for (uint32_t e = threadIdx.x; e < n; e += blockDim.x)
      st_s(sm + 2 * e, ntt_mul(ld_s(sm + 2 * e), ld_tab(a.tab, which == 0 ? QGR_LO : QG_LO, rev(e, a.lg))));
    __syncthreads();
    ntt_smem<false>(sm, 1, a.lg, n, a.tab, ROOT);
#pragma unroll 1
    for (uint32_t e = threadIdx.x; e < n; e += blockDim.x) {
      const fe y = ld_s(sm + 2 * e);
      if (which == 0) st_s(row + 2 * e, y);
      else if (which == 1) st_s(row + 2 * e, ntt_mul(y, ld_s(row + 2 * e)));
      else st_s(row + 2 * e, fe_sub(ld_s(row + 2 * e), y));
    }
    __syncthreads();
  }
}

// Column pass of n = n1 * n2 > 2^12: CTA = C adjacent columns of one vector (standalone) or of one row's A, B and C
// (QUOT), column c at shared entry c * (n2 + 1) (the pad spreads the C lanes of a row over the banks).
//   !QUOT: first pass.  Input reduced, times g^i (forward coset), DIF, times w_n^(+-i1 rev(p)), stored in place.
//   QUOT:  last pass of the quotient.  Times w_n^(i1 rev(p)), DIT (natural out), combined into the A slot as in
//          ntt_small_quotient_kernel.
template <bool QUOT>
__global__ void __launch_bounds__(NTT_THREADS, 2) ntt_col_kernel(const NttArgs a) {
  extern __shared__ uint4 sm[];
  const uint32_t n1 = 1u << a.lg1, n2 = 1u << a.lg2, C = a.C, stride = n2 + 1, lgC = 31 - __clz(C);
  const uint32_t groups = n1 >> lgC;
  const unsigned long long q = blockIdx.x / groups;
  const uint32_t col0 = (blockIdx.x % groups) * C;
  const bool inv = a.flags & NTT_INVERSE, coset = a.flags & NTT_COSET;
#pragma unroll 1
  for (uint32_t which = 0; which < (QUOT ? 3u : 1u); which++) {
    uint4* v = QUOT ? vec_ptr(a, 3 * q + which) : vec_ptr(a, q);
#pragma unroll 1
    for (uint32_t e = threadIdx.x; e < (C << a.lg2); e += blockDim.x) {
      const uint32_t c = e & (C - 1), p = e >> lgC, i1 = col0 + c;
      fe x = ld_s(v + 2 * ((size_t)p * n1 + i1));
      if (QUOT) x = mul_pow(x, a.tab, TW_LO, TW_HI, i1 * rev(p, a.lg2));
      else {
        x = reduce_in(x);
        if (coset && !inv) x = mul_pow(x, a.tab, CG_LO, CG_HI, i1 + p * n1);
      }
      st_s(sm + 2 * (c * stride + p), x);
    }
    __syncthreads();
    if (QUOT) ntt_smem<false>(sm, C, a.lg2, stride, a.tab, ROOT);
    else ntt_smem<true>(sm, C, a.lg2, stride, a.tab, inv ? IROOT : ROOT);
#pragma unroll 1
    for (uint32_t e = threadIdx.x; e < (C << a.lg2); e += blockDim.x) {
      const uint32_t c = e & (C - 1), p = e >> lgC, i1 = col0 + c;
      fe y = ld_s(sm + 2 * (c * stride + p));
      uint4* dst = vec_ptr(a, QUOT ? 3 * q : q) + 2 * ((size_t)p * n1 + i1);
      if (!QUOT) y = mul_pow(y, a.tab, inv ? ITW_LO : TW_LO, inv ? ITW_HI : TW_HI, i1 * rev(p, a.lg2));
      else if (which == 1) y = ntt_mul(y, ld_s(dst));
      else if (which == 2) y = fe_sub(ld_s(dst), y);
      st_s(dst, y);
    }
    __syncthreads();
  }
}

// Row pass of n = n1 * n2 > 2^12: CTA = C contiguous blocks of n1 entries of one vector.
//   !QUOT: DIF; entry P then holds y[rev_n(P)], times n^-1 (g^-rev_n(P)) for the inverse (coset).
//   QUOT:  inverse DIF, times n^-1 g^rev_n(P) (pre-scaled for A), forward DIT.
template <bool QUOT>
__global__ void __launch_bounds__(NTT_THREADS, 2) ntt_row_kernel(const NttArgs a) {
  extern __shared__ uint4 sm[];
  const uint32_t n1 = 1u << a.lg1, C = a.C, lgC = 31 - __clz(C), groups = (1u << a.lg2) >> lgC;
  const unsigned long long q = blockIdx.x / groups;
  const uint32_t P0 = (blockIdx.x % groups) * C * n1;
  uint4* v = vec_ptr(a, q) + 2 * (size_t)P0;
  const bool inv = QUOT || (a.flags & NTT_INVERSE), coset = a.flags & NTT_COSET;
#pragma unroll 1
  for (uint32_t e = threadIdx.x; e < (C << a.lg1); e += blockDim.x) st_s(sm + 2 * e, ld_s(v + 2 * e));
  __syncthreads();
  ntt_smem<true>(sm, C, a.lg1, n1, a.tab, inv ? IROOT : ROOT);
#pragma unroll 1
  for (uint32_t e = threadIdx.x; e < (C << a.lg1); e += blockDim.x) {
    fe y = ld_s(sm + 2 * e);
    const uint32_t i = rev(P0 + e, a.lg);
    if (QUOT) y = mul_pow(y, a.tab, q % 3 == 0 ? QGR_LO : QG_LO, CG_HI, i);
    else if (inv && coset) y = mul_pow(y, a.tab, ICG_LO, ICG_HI, i);
    else if (inv) y = ntt_mul(y, ld_tab(a.tab, NINV, 0));
    if (QUOT) st_s(sm + 2 * e, y);
    else st_s(v + 2 * e, y);
  }
  if (!QUOT) return;
  __syncthreads();
  ntt_smem<false>(sm, C, a.lg1, n1, a.tab, ROOT);
#pragma unroll 1
  for (uint32_t e = threadIdx.x; e < (C << a.lg1); e += blockDim.x) st_s(v + 2 * e, ld_s(sm + 2 * e));
}

// Bit-reversal permutation of vectors of 2^lg entries (lg >= 13), in place.  Entry (a, m, b) = a 2^(lg-4) + m 2^4 + b
// and its image (rev4 b, rev m, rev4 a): the CTA of m <= rev(m) swaps the 16 x 16 tiles of m and rev(m).
__global__ void __launch_bounds__(NTT_THREADS) ntt_bitrev_kernel(const NttArgs a) {
  __shared__ uint4 t0[2 * 256], t1[2 * 256];
  const uint32_t lgm = a.lg - 8, mids = 1u << lgm;
  const unsigned long long q = blockIdx.x / mids;
  const uint32_t m = blockIdx.x % mids, m2 = rev(m, lgm);
  if (m > m2) return;
  uint4* v = vec_ptr(a, q);
  const uint32_t e = threadIdx.x, hi = e >> 4, lo = e & 15;
  auto at = [&](uint32_t mm, uint32_t x, uint32_t y) { return v + 2 * (((size_t)x << (a.lg - 4)) + (mm << 4) + y); };
  st_s(t0 + 2 * e, ld_s(at(m, hi, lo)));
  st_s(t1 + 2 * e, ld_s(at(m2, hi, lo)));
  __syncthreads();
  const uint32_t src = (rev(lo, 4) << 4) + rev(hi, 4);
  st_s(at(m, hi, lo), ld_s(t1 + 2 * src));
  if (m != m2) st_s(at(m2, hi, lo), ld_s(t0 + 2 * src));
}

namespace {

std::mutex g_mu;
std::map<int, bool> g_ready;                          // kernel attributes set on this device
std::map<std::pair<int, uint32_t>, uint4*> g_tabs;    // (device, log_n) -> ntt_build_tables(log_n), process lifetime

// the twiddle tables of 2^lg on `device` (built and uploaded on first use; 1.6 MB each)
const uint4* ntt_tables(int device, uint32_t lg) {
  std::lock_guard<std::mutex> lk(g_mu);
  auto it = g_tabs.find({device, lg});
  if (it != g_tabs.end()) return it->second;
  check_device(device);
  DeviceGuard on(device);
  if (!g_ready[device]) {
    cudaDeviceProp prop; CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
    const int smem = (int)prop.sharedMemPerBlockOptin;
    CUDA_CHECK(cudaFuncSetAttribute(ntt_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    CUDA_CHECK(cudaFuncSetAttribute(ntt_small_quotient_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    CUDA_CHECK(cudaFuncSetAttribute(ntt_col_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    CUDA_CHECK(cudaFuncSetAttribute(ntt_col_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    CUDA_CHECK(cudaFuncSetAttribute(ntt_row_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    CUDA_CHECK(cudaFuncSetAttribute(ntt_row_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    g_ready[device] = true;
  }
  const std::vector<fe> tab = ntt_build_tables(lg);
  uint4* d = nullptr;
  CUDA_CHECK(cudaMalloc(&d, tab.size() * 32));
  const cudaError_t e = cudaMemcpy(d, tab.data(), tab.size() * 32, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { cudaFree(d); CUDA_CHECK(e); }
  g_tabs[{device, lg}] = d;
  return d;
}

NttArgs ntt_args(int device, void* d, unsigned long long pitch, uint32_t per_row, unsigned long long n_vectors, uint32_t lg,
                 uint32_t flags) {
  NttArgs a;
  a.base = (uint8_t*)d; a.pitch = pitch; a.vec_b = 32ull << lg; a.per_row = per_row; a.n_vectors = n_vectors;
  a.lg = lg; a.lg2 = lg / 2; a.lg1 = lg - a.lg2; a.flags = flags;
  a.tab = ntt_tables(device, lg);
  return a;
}

unsigned grid_of(unsigned long long blocks) {
  if (blocks > 0x7FFFFFFFull) throw Error("ntt: batch too large (more than 2^31 - 1 CTAs)");
  return (unsigned)blocks;
}

// the two passes of n > 2^12; C sub-transforms per CTA for each
void ntt_two_pass(NttArgs a, unsigned long long vectors, bool quot, cudaStream_t s) {
  const uint32_t col_c = std::min<uint32_t>(1u << a.lg1, std::max<uint32_t>(1, NTT_CTA_ELEMS >> a.lg2));
  const uint32_t row_c = std::min<uint32_t>(1u << a.lg2, std::max<uint32_t>(1, NTT_CTA_ELEMS >> a.lg1));
  NttArgs c = a, r = a;
  c.C = col_c; r.C = row_c;
  const size_t col_smem = (size_t)col_c * ((1u << a.lg2) + 1) * 32, row_smem = ((size_t)row_c << a.lg1) * 32;
  const unsigned long long rows = quot ? vectors / 3 : vectors;
  if (!quot) {
    ntt_col_kernel<false><<<grid_of(rows * ((1u << a.lg1) / col_c)), NTT_THREADS, col_smem, s>>>(c);
    CUDA_CHECK(cudaGetLastError());
    ntt_row_kernel<false><<<grid_of(vectors * ((1u << a.lg2) / row_c)), NTT_THREADS, row_smem, s>>>(r);
    CUDA_CHECK(cudaGetLastError());
    ntt_bitrev_kernel<<<grid_of(vectors << (a.lg - 8)), NTT_THREADS, 0, s>>>(a);
    CUDA_CHECK(cudaGetLastError());
    return;
  }
  // quotient: inverse DIF column pass on A, B and C, then the fused row pass, then the combining DIT column pass
  NttArgs ci = c;
  ci.flags = NTT_INVERSE;
  ntt_col_kernel<false><<<grid_of(vectors * ((1u << a.lg1) / col_c)), NTT_THREADS, col_smem, s>>>(ci);
  CUDA_CHECK(cudaGetLastError());
  ntt_row_kernel<true><<<grid_of(vectors * ((1u << a.lg2) / row_c)), NTT_THREADS, row_smem, s>>>(r);
  CUDA_CHECK(cudaGetLastError());
  ntt_col_kernel<true><<<grid_of(rows * ((1u << a.lg1) / col_c)), NTT_THREADS, col_smem, s>>>(c);
  CUDA_CHECK(cudaGetLastError());
}

}  // namespace

size_t ntt_check_args(const void* d_data, uint32_t log_n, size_t pitch, uint32_t flags) {
  if (flags & ~(NTT_INVERSE | NTT_COSET))
    throw Error("unknown flag bits " + std::to_string(flags & ~(NTT_INVERSE | NTT_COSET)) + " (known: GW_NTT_INVERSE, GW_NTT_COSET)");
  if (log_n > NTT_MAX_LOG)
    throw Error("log_n = " + std::to_string(log_n) + " is larger than 24: domains above 2^24 are not supported");
  const size_t vec_b = (size_t)32 << log_n;
  if (pitch == 0) pitch = vec_b;
  if (pitch < vec_b) throw Error("pitch is smaller than 2^log_n x 32 bytes");
  if (pitch % 16) throw Error("pitch must be a multiple of 16");
  if ((uintptr_t)d_data & 15) throw Error("device buffers must be 16-byte aligned");
  return pitch;
}

void ntt_batch_device(int device, void* d_data, size_t n_vectors, uint32_t log_n, size_t pitch, uint32_t flags, void* stream) {
  pitch = ntt_check_args(d_data, log_n, pitch, flags);
  if (n_vectors == 0) return;
  NttArgs a = ntt_args(device, d_data, pitch, 1, n_vectors, log_n, flags);
  DeviceGuard on(device);
  cudaStream_t s = (cudaStream_t)stream;
  if (log_n <= 12) {
    a.C = std::max<uint32_t>(1, NTT_CTA_ELEMS >> log_n);
    ntt_small_kernel<<<grid_of((n_vectors + a.C - 1) / a.C), NTT_THREADS, ((size_t)a.C << log_n) * 32, s>>>(a);
    CUDA_CHECK(cudaGetLastError());
    return;
  }
  ntt_two_pass(a, n_vectors, false, s);
}

void ntt_quotient_device(int device, void* d_work, size_t B, uint32_t log_n, size_t pitch, void* stream) {
  if (log_n > NTT_MAX_LOG)
    throw Error("the Groth16 domain 2^" + std::to_string(log_n) + " is larger than 2^24: domains above 2^24 are not supported");
  if (B == 0) return;
  NttArgs a = ntt_args(device, d_work, pitch, 3, 3 * (unsigned long long)B, log_n, 0);
  DeviceGuard on(device);
  cudaStream_t s = (cudaStream_t)stream;
  if (log_n <= 12) {
    a.C = 1;
    ntt_small_quotient_kernel<<<grid_of(B), NTT_THREADS, (size_t)32 << log_n, s>>>(a);
    CUDA_CHECK(cudaGetLastError());
    return;
  }
  ntt_two_pass(a, 3 * (unsigned long long)B, true, s);
}

}  // namespace gw
