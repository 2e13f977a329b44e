// Device twin of field_host_api.cpp: every primitive of csrc/field.cuh, csrc/inv_safegcd.cuh, csrc/alu.cuh and the
// butterflies of csrc/ntt.cuh run on the GPU over arrays of operand tuples, so that pytest can check the code the kernels
// actually run (the PTX carry chains, __funnelshift_r, carries kept between asm statements) against Python integers.
//
// One thread evaluates one tuple.  Each primitive is its own kernel, a template instance, so the primitive is inlined
// and register-allocated on its own the way the engine's kernels inline it, and each is built twice: "roomy" (128
// threads, no register limit) and "starved" (__launch_bounds__(1024, 2): at most 32 registers, so the carry chains
// spill to local memory).  fd_launch never aborts: it returns the first CUDA error.
#include <cuda_runtime.h>
#include <string.h>

#include "../../circom-witnesscalc_b200/csrc/alu.cuh"
#include "../../circom-witnesscalc_b200/csrc/ntt.cuh"

using namespace gw;

namespace {

// primitive ids; tests/test_gpu_field.py names them in this order
enum Prim : int {
  P_MUL, P_MUL_WIDE, P_SQR_WIDE, P_SQR, P_MUL_LO, P_MONT_MUL, P_TO_MONT, P_FROM_MONT, P_ADD, P_SUB, P_NEG, P_REDUCE,
  P_SHR, P_SHL, P_BITOP, P_BNOT, P_CMP, P_DIVREM, P_POW, P_INV_FERMAT, P_INV_SAFEGCD, P_MUL_HI_TRUNC, P_MONT_REDUCE,
  P_DOT_EVAL, P_MUL2, P_NTT_MUL, P_BFLY_DIF, P_BFLY_DIT, P_ALU, P_FROM_NARROW, N_PRIM
};
// 32-bit words per row of the operand arrays a, b, c and of the output; op and status are one word per row
struct Shape { int a, b, c, out; };
constexpr int DOT_TERMS = 16;   // isa.h DOT_MAX_TERMS
constexpr Shape SHAPES[N_PRIM] = {
    {8, 8, 0, 8}, {8, 8, 0, 16}, {8, 0, 0, 16}, {8, 0, 0, 8}, {8, 8, 0, 8}, {8, 8, 0, 8}, {8, 0, 0, 8}, {8, 0, 0, 8},
    {8, 8, 0, 8}, {8, 8, 0, 8}, {8, 0, 0, 8}, {8, 0, 0, 8},
    {8, 8, 0, 8}, {8, 8, 0, 8}, {8, 8, 0, 8}, {8, 0, 0, 8}, {8, 8, 0, 0}, {8, 8, 0, 16}, {8, 8, 0, 8}, {8, 0, 0, 8},
    {8, 0, 0, 8}, {8, 8, 0, 16}, {16, 0, 0, 8},
    {8 * DOT_TERMS, 8 * DOT_TERMS, 1, 8}, {16, 16, 0, 16}, {8, 8, 0, 8}, {8, 8, 8, 16}, {8, 8, 8, 16}, {8, 8, 8, 8},
    {2, 0, 0, 8},
};

struct Args {
  int n;
  const uint32_t *a, *b, *c, *op;
  uint32_t *out, *status;
};

__device__ __forceinline__ fe ld(const uint32_t* p) { fe r; for (int i = 0; i < 8; i++) r.l[i] = p[i]; return r; }
__device__ __forceinline__ void st(uint32_t* p, const fe& v) { for (int i = 0; i < 8; i++) p[i] = v.l[i]; }

template <int P> __device__ __forceinline__ void body(const Args& g, int t) {
  constexpr Shape S = SHAPES[P];
  const uint32_t* a = g.a + (size_t)t * S.a;
  const uint32_t* b = g.b + (size_t)t * S.b;
  const uint32_t* c = g.c + (size_t)t * S.c;
  uint32_t* o = g.out + (size_t)t * S.out;
  const uint32_t op = g.op[t];
  uint32_t s = 0;
  if constexpr (P == P_MUL) st(o, fe_mul(ld(a), ld(b)));
  else if constexpr (P == P_MUL_WIDE) { uint32_t r[16], x[8], y[8]; for (int i = 0; i < 8; i++) { x[i] = a[i]; y[i] = b[i]; } u256_mul_wide(r, x, y); for (int i = 0; i < 16; i++) o[i] = r[i]; }
  else if constexpr (P == P_SQR_WIDE) { uint32_t r[16], x[8]; for (int i = 0; i < 8; i++) x[i] = a[i]; u256_sqr_wide(r, x); for (int i = 0; i < 16; i++) o[i] = r[i]; }
  else if constexpr (P == P_SQR) st(o, fe_sqr(ld(a)));
  else if constexpr (P == P_MUL_LO) { uint32_t r[8], x[8], y[8]; for (int i = 0; i < 8; i++) { x[i] = a[i]; y[i] = b[i]; } u256_mul_lo(r, x, y); for (int i = 0; i < 8; i++) o[i] = r[i]; }
  else if constexpr (P == P_MONT_MUL) st(o, fe_mont_mul(ld(a), ld(b)));
  else if constexpr (P == P_TO_MONT) st(o, fe_to_mont(ld(a)));
  else if constexpr (P == P_FROM_MONT) st(o, fe_from_mont(ld(a)));
  else if constexpr (P == P_ADD) st(o, fe_add(ld(a), ld(b)));
  else if constexpr (P == P_SUB) st(o, fe_sub(ld(a), ld(b)));
  else if constexpr (P == P_NEG) st(o, fe_neg(ld(a)));
  else if constexpr (P == P_REDUCE) st(o, fe_reduce256(ld(a)));
  else if constexpr (P == P_SHR) st(o, fe_shr(ld(a), ld(b)));
  else if constexpr (P == P_SHL) { bool ov; st(o, fe_shl(ld(a), ld(b), &ov)); s = ov; }
  else if constexpr (P == P_BITOP) { bool eq; st(o, fe_bitop(ld(a), ld(b), (int)op, &eq)); s = eq; }
  else if constexpr (P == P_BNOT) st(o, fe_bnot(ld(a)));
  else if constexpr (P == P_CMP) s = fe_cmp(ld(a), ld(b), (int)op);
  else if constexpr (P == P_DIVREM) { fe q, r; u256_divrem(ld(a), ld(b), &q, &r); st(o, q); st(o + 8, r); }
  else if constexpr (P == P_POW) st(o, fe_pow(ld(a), ld(b)));
  else if constexpr (P == P_INV_FERMAT) st(o, fe_inv_fermat(ld(a)));
  else if constexpr (P == P_INV_SAFEGCD) st(o, fe_inv(ld(a)));
  else if constexpr (P == P_MUL_HI_TRUNC) { uint32_t r[16], x[8], y[8]; for (int i = 0; i < 8; i++) { x[i] = a[i]; y[i] = b[i]; } u256_mul_hi_trunc(r, x, y); for (int i = 0; i < 16; i++) o[i] = r[i]; }
  else if constexpr (P == P_MONT_REDUCE) { uint32_t p16[16]; for (int i = 0; i < 16; i++) p16[i] = a[i]; dot_acc A; dot_load(A, p16); st(o, fe_mont_reduce(A, (int)op)); }
  else if constexpr (P == P_DOT_EVAL) {
    // the term loop of engine.cu (eval_batch_kernel, OP_DOT): kinds read at run time, not unrolled.  op: 2 bits of kind
    // per term; c[0]: n_terms | n_cond_sub << 8
    const uint32_t nt = c[0] & 0xFFu;
    dot_acc A;
    dot_init(A);
#pragma unroll 1
    for (uint32_t k = 0; k < nt; k++) {
      const uint32_t kind = (op >> (2 * k)) & 3u;
      if (kind == T_MAC) {
        const fe cv = ld(b + 8 * k);
        const fe x = ld(a + 8 * k);
        dot_mac(A, x.l, cv.l);
      } else if (kind == T_CONST) {
        const fe cv = ld(b + 8 * k);
        dot_add256(A, cv.l, 0);
      } else {
        dot_term(A, kind, ld(a + 8 * k), fe_zero());
      }
    }
    st(o, fe_mont_reduce(A, (int)((c[0] >> 8) & 0xFFu)));
  }
  else if constexpr (P == P_MUL2) { fe r1, r2; fe_mul2(ld(a), ld(b), ld(a + 8), ld(b + 8), r1, r2); st(o, r1); st(o + 8, r2); }
  else if constexpr (P == P_NTT_MUL) st(o, ntt_mul(ld(a), ld(b)));
  else if constexpr (P == P_BFLY_DIF) { fe x = ld(a), y = ld(b); ntt_bfly_dif(x, y, ld(c)); st(o, x); st(o + 8, y); }
  else if constexpr (P == P_BFLY_DIT) { fe x = ld(a), y = ld(b); ntt_bfly_dit(x, y, ld(c)); st(o, x); st(o + 8, y); }
  else if constexpr (P == P_ALU) st(o, alu_exec(op, ld(a), ld(b), ld(c), s));
  else if constexpr (P == P_FROM_NARROW) st(o, fe_from_narrow((int64_t)((uint64_t)a[0] | ((uint64_t)a[1] << 32))));
  g.status[t] = s;
}

template <int P> __global__ void roomy_kernel(Args g) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < g.n) body<P>(g, t);
}
template <int P> __global__ void __launch_bounds__(1024, 2) starved_kernel(Args g) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < g.n) body<P>(g, t);
}

constexpr int ROOMY_THREADS = 128, STARVED_THREADS = 1024;

template <int P> cudaError_t launch(int prim, int variant, const Args& g) {
  if constexpr (P == N_PRIM) {
    return cudaErrorInvalidValue;
  } else {
    if (prim != P) return launch<P + 1>(prim, variant, g);
    if (variant == 0) roomy_kernel<P><<<(g.n + ROOMY_THREADS - 1) / ROOMY_THREADS, ROOMY_THREADS>>>(g);
    else starved_kernel<P><<<(g.n + STARVED_THREADS - 1) / STARVED_THREADS, STARVED_THREADS>>>(g);
    return cudaGetLastError();
  }
}

// device copies of the cap rows of one array
struct Buf {
  uint32_t* d = nullptr;
  size_t bytes = 0;
  cudaError_t up(const uint32_t* h, size_t words) {
    bytes = words * 4;
    if (!bytes) return cudaSuccess;
    cudaError_t e = cudaMalloc(&d, bytes);
    if (e == cudaSuccess) e = cudaMemcpy(d, h, bytes, cudaMemcpyHostToDevice);
    return e;
  }
  cudaError_t down(uint32_t* h) const { return bytes ? cudaMemcpy(h, d, bytes, cudaMemcpyDeviceToHost) : cudaSuccess; }
  ~Buf() { if (d) cudaFree(d); }
};

}  // namespace

extern "C" {

int fd_n_prims(void) { return N_PRIM; }

// words per row of a, b, c and out of primitive `prim`; -1 for an unknown id
int fd_shape(int prim, int* words4) {
  if (prim < 0 || prim >= N_PRIM) return -1;
  words4[0] = SHAPES[prim].a; words4[1] = SHAPES[prim].b; words4[2] = SHAPES[prim].c; words4[3] = SHAPES[prim].out;
  return 0;
}

// Rows 0 .. n - 1 of primitive `prim` in variant 0 (roomy) or 1 (starved).  Every array holds cap >= n rows (fd_shape);
// all cap rows of out and status go to the device and come back, so rows from n on must come back as they were sent.
// Returns the first cudaError_t (0 on success).
int fd_launch(int prim, int variant, int n, int cap, const uint32_t* a, const uint32_t* b, const uint32_t* c,
              const uint32_t* op, uint32_t* out, uint32_t* status) {
  if (prim < 0 || prim >= N_PRIM || variant < 0 || variant > 1 || n < 0 || cap < n) return (int)cudaErrorInvalidValue;
  const Shape S = SHAPES[prim];
  const size_t rows = (size_t)cap;
  Buf A, B, C, OP, OUT, ST;
  cudaError_t e = A.up(a, rows * S.a);
  if (e == cudaSuccess) e = B.up(b, rows * S.b);
  if (e == cudaSuccess) e = C.up(c, rows * S.c);
  if (e == cudaSuccess) e = OP.up(op, rows);
  if (e == cudaSuccess) e = OUT.up(out, rows * S.out);
  if (e == cudaSuccess) e = ST.up(status, rows);
  if (e == cudaSuccess && n > 0) e = launch<0>(prim, variant, Args{n, A.d, B.d, C.d, OP.d, OUT.d, ST.d});
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = OUT.down(out);
  if (e == cudaSuccess) e = ST.down(status);
  return (int)e;
}

}  // extern "C"
