// BN254 scalar-field and 256-bit integer arithmetic on 8 x 32-bit limbs (little-endian limbs).
//
// Replaces, on the device, what the reference gets from ark-ff / ruint behind
// /root/reference/src/graph.rs:102-144 (Operation::eval_fr), :188-197, :221-225 and the helpers
// :621-769 (shl, shr, bit_and/or/xor, u_lt/u_gt/u_lte/u_gte), modulus from src/field.rs:3-4.
//
// Design choice (see DESIGN.md "value domain"): graph values are kept CANONICAL in [0, M), not in
// Montgomery form.  Multiplication is schoolbook 8x8 + Barrett reduction (q = floor(ab/M) estimated
// from the top 256 bits with mu = floor(2^509/M); the estimate is never more than 1 too small).
// The integer-domain ops (shifts, bitwise, comparisons, Idiv/Mod) and the .wtns output then need no
// Montgomery<->canonical conversion at all, which is where the reference spends most of its time on
// bit-heavy graphs.  Montgomery multiplication (fe_mont_mul) is provided for chains that stay in the
// field (inversion, pow).
//
// Every function is __host__ __device__: the device path uses PTX carry chains
// (mad.lo.cc / madc.hi.cc pairs that ptxas fuses into IMAD.WIDE.U32 with carry), the host path is
// plain C used only by the unit tests of this header (tests/csrc/test_field_host.cpp).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define GW_HD __host__ __device__ __forceinline__
#define GW_HD_NOINLINE inline __host__ __device__ __noinline__   // inline: one definition however many .cu files include this
#else
#define GW_HD inline
#define GW_HD_NOINLINE inline __attribute__((noinline))
#endif

namespace gw {

struct fe { uint32_t l[8]; };

// ---- constants (constexpr selectors so that unrolled device code sees immediates) ---------------
GW_HD constexpr uint32_t MOD_L(int i) {   // M
  return i == 0 ? 0xf0000001u : i == 1 ? 0x43e1f593u : i == 2 ? 0x79b97091u : i == 3 ? 0x2833e848u :
         i == 4 ? 0x8181585du : i == 5 ? 0xb85045b6u : i == 6 ? 0xe131a029u : 0x30644e72u;
}
GW_HD constexpr uint32_t MU_L(int i) {    // floor(2^509 / M)
  return i == 0 ? 0x7c3bd24bu : i == 1 ? 0xc40e074du : i == 2 ? 0x13d1015cu : i == 3 ? 0xe2890a40u :
         i == 4 ? 0xd00e6028u : i == 5 ? 0x560e94b0u : i == 6 ? 0xc474094fu : 0xa948e8c4u;
}
GW_HD constexpr uint32_t HALF_L(int i) {  // floor(M / 2), graph.rs:720
  return i == 0 ? 0xf8000000u : i == 1 ? 0xa1f0fac9u : i == 2 ? 0x3cdcb848u : i == 3 ? 0x9419f424u :
         i == 4 ? 0x40c0ac2eu : i == 5 ? 0xdc2822dbu : i == 6 ? 0x7098d014u : 0x18322739u;
}
GW_HD constexpr uint32_t MM2_L(int i) {   // M - 2 (Fermat exponent)
  return i == 0 ? 0xefffffffu : MOD_L(i);
}
GW_HD constexpr uint32_t R2_L(int i) {    // 2^512 mod M
  return i == 0 ? 0xae216da7u : i == 1 ? 0x1bb8e645u : i == 2 ? 0xe35c59e3u : i == 3 ? 0x53fe3ab1u :
         i == 4 ? 0x53bb8085u : i == 5 ? 0x8c49833du : i == 6 ? 0x7f4e44a5u : 0x0216d0b1u;
}
GW_HD constexpr uint32_t R1_L(int i) {    // 2^256 mod M
  return i == 0 ? 0x4ffffffbu : i == 1 ? 0xac96341cu : i == 2 ? 0x9f60cd29u : i == 3 ? 0x36fc7695u :
         i == 4 ? 0x7879462eu : i == 5 ? 0x666ea36fu : i == 6 ? 0x9a07df2fu : 0x0e0a77c1u;
}
GW_HD constexpr uint32_t MODS_L(int i, int s) {   // limb i of M << s, s in {0, 1, 2}  (4M < 2^256)
  return s == 0 ? MOD_L(i) : ((MOD_L(i) << s) | (i > 0 ? (MOD_L(i - 1) >> (32 - s)) : 0u));
}
static const uint32_t MONT_INV32 = 0xefffffffu;   // -M^-1 mod 2^32

GW_HD fe fe_zero() { fe r; for (int i = 0; i < 8; i++) r.l[i] = 0; return r; }
GW_HD fe fe_small(uint32_t v) { fe r = fe_zero(); r.l[0] = v; return r; }
GW_HD fe fe_modulus() { fe r; for (int i = 0; i < 8; i++) r.l[i] = MOD_L(i); return r; }

// ---- carry-chain primitives ----------------------------------------------------------------------
// GW_CHAINS: the carry-chain formulations below are compiled (device code, or the host emulation of the PTX carry flag
// used by the unit tests: -DGW_EMULATE_PTX runs the DEVICE algorithms on the CPU, instruction for instruction)
#if defined(__CUDA_ARCH__) || defined(GW_EMULATE_PTX)
#define GW_CHAINS 1
#endif
#if !defined(__CUDA_ARCH__) && defined(GW_EMULATE_PTX)
static thread_local uint32_t gw_cf = 0;     // the PTX condition-code carry flag
inline uint32_t ptx_add_cc(uint32_t a, uint32_t b) { uint64_t t = (uint64_t)a + b; gw_cf = (uint32_t)(t >> 32); return (uint32_t)t; }
inline uint32_t ptx_addc_cc(uint32_t a, uint32_t b) { uint64_t t = (uint64_t)a + b + gw_cf; gw_cf = (uint32_t)(t >> 32); return (uint32_t)t; }
inline uint32_t ptx_addc(uint32_t a, uint32_t b) { return a + b + gw_cf; }
inline uint32_t ptx_sub_cc(uint32_t a, uint32_t b) { uint64_t t = (uint64_t)a - b; gw_cf = (uint32_t)(t >> 32) & 1u; return (uint32_t)t; }   // CF = borrow here
inline uint32_t ptx_subc_cc(uint32_t a, uint32_t b) { uint64_t t = (uint64_t)a - b - gw_cf; gw_cf = (uint32_t)(t >> 32) & 1u; return (uint32_t)t; }
inline uint32_t ptx_subc(uint32_t a, uint32_t b) { return a - b - gw_cf; }
inline uint32_t ptx_mad_lo_cc(uint32_t a, uint32_t b, uint32_t c) { uint64_t t = (uint64_t)(uint32_t)((uint64_t)a * b) + c; gw_cf = (uint32_t)(t >> 32); return (uint32_t)t; }
inline uint32_t ptx_madc_lo_cc(uint32_t a, uint32_t b, uint32_t c) { uint64_t t = (uint64_t)(uint32_t)((uint64_t)a * b) + c + gw_cf; gw_cf = (uint32_t)(t >> 32); return (uint32_t)t; }
inline uint32_t ptx_mad_hi_cc(uint32_t a, uint32_t b, uint32_t c) { uint64_t t = (((uint64_t)a * b) >> 32) + c; gw_cf = (uint32_t)(t >> 32); return (uint32_t)t; }
inline uint32_t ptx_madc_hi_cc(uint32_t a, uint32_t b, uint32_t c) { uint64_t t = (((uint64_t)a * b) >> 32) + c + gw_cf; gw_cf = (uint32_t)(t >> 32); return (uint32_t)t; }
inline uint32_t ptx_madc_hi(uint32_t a, uint32_t b, uint32_t c) { return (uint32_t)((((uint64_t)a * b) >> 32) + c + gw_cf); }
#endif
#if defined(__CUDA_ARCH__)
#define GW_ASM asm volatile
__device__ __forceinline__ uint32_t ptx_add_cc(uint32_t a, uint32_t b) { uint32_t r; GW_ASM("add.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
__device__ __forceinline__ uint32_t ptx_addc_cc(uint32_t a, uint32_t b) { uint32_t r; GW_ASM("addc.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
__device__ __forceinline__ uint32_t ptx_addc(uint32_t a, uint32_t b) { uint32_t r; GW_ASM("addc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
__device__ __forceinline__ uint32_t ptx_sub_cc(uint32_t a, uint32_t b) { uint32_t r; GW_ASM("sub.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
__device__ __forceinline__ uint32_t ptx_subc_cc(uint32_t a, uint32_t b) { uint32_t r; GW_ASM("subc.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
__device__ __forceinline__ uint32_t ptx_subc(uint32_t a, uint32_t b) { uint32_t r; GW_ASM("subc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
__device__ __forceinline__ uint32_t ptx_mad_lo_cc(uint32_t a, uint32_t b, uint32_t c) { uint32_t r; GW_ASM("mad.lo.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r; }
__device__ __forceinline__ uint32_t ptx_madc_lo_cc(uint32_t a, uint32_t b, uint32_t c) { uint32_t r; GW_ASM("madc.lo.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r; }
__device__ __forceinline__ uint32_t ptx_mad_hi_cc(uint32_t a, uint32_t b, uint32_t c) { uint32_t r; GW_ASM("mad.hi.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r; }
__device__ __forceinline__ uint32_t ptx_madc_hi_cc(uint32_t a, uint32_t b, uint32_t c) { uint32_t r; GW_ASM("madc.hi.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r; }
__device__ __forceinline__ uint32_t ptx_madc_hi(uint32_t a, uint32_t b, uint32_t c) { uint32_t r; GW_ASM("madc.hi.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r; }
#endif

// Pair accumulators.  One (mad.lo.cc, madc.hi.cc) pair becomes ONE IMAD.WIDE.U32(.X) whose 64-bit addend and result
// are an aligned register pair.  Accumulators that live across a loop (the OP_DOT term loop) are therefore kept as
// 64-bit values: with separate 32-bit registers ptxas re-pairs them around every loop iteration (measured on the
// authV2 kernel, profiles/r02b: 37 IMAD.MOV.U32 next to the 64 IMAD.WIDE of one dot_mac -- moves that sit on the same
// pipe as the multiplications).  acc = {lo = column c, hi = column c + 1}.
#if defined(GW_CHAINS)
#if defined(__CUDA_ARCH__)
__device__ __forceinline__ void ptx_mac64_first(uint64_t& acc, uint32_t a, uint32_t b) {      // acc += a*b; CF = carry out
  GW_ASM("{\n\t.reg .u32 l, h;\n\tmov.b64 {l, h}, %0;\n\tmad.lo.cc.u32 l, %1, %2, l;\n\tmadc.hi.cc.u32 h, %1, %2, h;\n\tmov.b64 %0, {l, h};\n\t}" : "+l"(acc) : "r"(a), "r"(b));
}
__device__ __forceinline__ void ptx_mac64_next(uint64_t& acc, uint32_t a, uint32_t b) {       // acc += a*b + CF; CF = carry out
  GW_ASM("{\n\t.reg .u32 l, h;\n\tmov.b64 {l, h}, %0;\n\tmadc.lo.cc.u32 l, %1, %2, l;\n\tmadc.hi.cc.u32 h, %1, %2, h;\n\tmov.b64 %0, {l, h};\n\t}" : "+l"(acc) : "r"(a), "r"(b));
}
__device__ __forceinline__ void ptx_machi64_first(uint64_t& acc, uint32_t a, uint32_t b) {    // hi half += hi(a*b); CF = carry out
  GW_ASM("{\n\t.reg .u32 l, h;\n\tmov.b64 {l, h}, %0;\n\tmad.hi.cc.u32 h, %1, %2, h;\n\tmov.b64 %0, {l, h};\n\t}" : "+l"(acc) : "r"(a), "r"(b));
}
__device__ __forceinline__ void ptx_add64_cc(uint64_t& acc, uint64_t v) { GW_ASM("add.cc.u64 %0, %0, %1;" : "+l"(acc) : "l"(v)); }
__device__ __forceinline__ void ptx_addc64_cc(uint64_t& acc, uint64_t v) { GW_ASM("addc.cc.u64 %0, %0, %1;" : "+l"(acc) : "l"(v)); }
#else
inline void ptx_mac64_first(uint64_t& acc, uint32_t a, uint32_t b) {
  const uint32_t l = ptx_mad_lo_cc(a, b, (uint32_t)acc), h = ptx_madc_hi_cc(a, b, (uint32_t)(acc >> 32));
  acc = (uint64_t)l | ((uint64_t)h << 32);
}
inline void ptx_mac64_next(uint64_t& acc, uint32_t a, uint32_t b) {
  const uint32_t l = ptx_madc_lo_cc(a, b, (uint32_t)acc), h = ptx_madc_hi_cc(a, b, (uint32_t)(acc >> 32));
  acc = (uint64_t)l | ((uint64_t)h << 32);
}
inline void ptx_machi64_first(uint64_t& acc, uint32_t a, uint32_t b) {
  const uint32_t h = ptx_mad_hi_cc(a, b, (uint32_t)(acc >> 32));
  acc = (acc & 0xFFFFFFFFull) | ((uint64_t)h << 32);
}
inline void ptx_add64_cc(uint64_t& acc, uint64_t v) {
  const uint32_t l = ptx_add_cc((uint32_t)acc, (uint32_t)v), h = ptx_addc_cc((uint32_t)(acc >> 32), (uint32_t)(v >> 32));
  acc = (uint64_t)l | ((uint64_t)h << 32);
}
inline void ptx_addc64_cc(uint64_t& acc, uint64_t v) {
  const uint32_t l = ptx_addc_cc((uint32_t)acc, (uint32_t)v), h = ptx_addc_cc((uint32_t)(acc >> 32), (uint32_t)(v >> 32));
  acc = (uint64_t)l | ((uint64_t)h << 32);
}
#endif
GW_HD uint64_t pair64(uint32_t lo, uint32_t hi) { return (uint64_t)lo | ((uint64_t)hi << 32); }
#endif

// r = a + b (mod 2^256); returns the carry out
GW_HD uint32_t u256_add(uint32_t* r, const uint32_t* a, const uint32_t* b) {
#if defined(GW_CHAINS)
  r[0] = ptx_add_cc(a[0], b[0]);
#pragma unroll
  for (int i = 1; i < 8; i++) r[i] = ptx_addc_cc(a[i], b[i]);
  return ptx_addc(0, 0);
#else
  uint64_t c = 0;
  for (int i = 0; i < 8; i++) { c += (uint64_t)a[i] + b[i]; r[i] = (uint32_t)c; c >>= 32; }
  return (uint32_t)c;
#endif
}

// r = a - b (mod 2^256); returns the borrow out (1 if a < b)
GW_HD uint32_t u256_sub(uint32_t* r, const uint32_t* a, const uint32_t* b) {
#if defined(GW_CHAINS)
  r[0] = ptx_sub_cc(a[0], b[0]);
#pragma unroll
  for (int i = 1; i < 8; i++) r[i] = ptx_subc_cc(a[i], b[i]);
  return ptx_subc(0, 0) & 1u;     // 0 - 0 - borrow = 0xFFFFFFFF when borrow
#else
  int64_t c = 0;
  for (int i = 0; i < 8; i++) { c += (int64_t)a[i] - b[i]; r[i] = (uint32_t)c; c >>= 32; }
  return (uint32_t)(c & 1);
#endif
}

GW_HD bool u256_is_zero(const uint32_t* a) {
  uint32_t o = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) o |= a[i];
  return o == 0;
}
GW_HD bool u256_eq(const uint32_t* a, const uint32_t* b) {
  uint32_t o = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) o |= a[i] ^ b[i];
  return o == 0;
}
// a < b (unsigned)
GW_HD bool u256_lt(const uint32_t* a, const uint32_t* b) {
  uint32_t t[8];
  return u256_sub(t, a, b) != 0;
}

// if a >= M then a -= M
GW_HD void fe_cond_sub_m(fe& a) {
  fe m = fe_modulus();
  uint32_t t[8];
  uint32_t borrow = u256_sub(t, a.l, m.l);
#pragma unroll
  for (int i = 0; i < 8; i++) a.l[i] = borrow ? a.l[i] : t[i];
}
// if a >= (M << S) then a -= (M << S)
template <int S> GW_HD void fe_cond_sub_ms(fe& a) {
  uint32_t m[8], t[8];
#pragma unroll
  for (int i = 0; i < 8; i++) m[i] = MODS_L(i, S);
  uint32_t borrow = u256_sub(t, a.l, m);
#pragma unroll
  for (int i = 0; i < 8; i++) a.l[i] = borrow ? a.l[i] : t[i];
}
GW_HD bool fe_is_zero(const fe& a) { return u256_is_zero(a.l); }
GW_HD bool fe_geq_m(const fe& a) { fe m = fe_modulus(); return !u256_lt(a.l, m.l); }

// any 256-bit integer -> [0, M)   (Fr::new / from_le_bytes_mod_order on load, graph.rs:376, storage.rs:28)
GW_HD fe fe_reduce256(fe a) {
#pragma unroll 1
  for (int k = 0; k < 5; k++) fe_cond_sub_m(a);   // 2^256 / M < 5.3
  return a;
}

GW_HD fe fe_add(const fe& a, const fe& b) {          // graph.rs:110
  fe r; u256_add(r.l, a.l, b.l);                     // a + b < 2M < 2^256: no carry out
  fe_cond_sub_m(r); return r;
}
GW_HD fe fe_sub(const fe& a, const fe& b) {          // graph.rs:111
  fe r; uint32_t borrow = u256_sub(r.l, a.l, b.l);
  fe m = fe_modulus(); uint32_t t[8]; u256_add(t, r.l, m.l);
#pragma unroll
  for (int i = 0; i < 8; i++) r.l[i] = borrow ? t[i] : r.l[i];
  return r;
}
GW_HD fe fe_neg(const fe& a) {                       // graph.rs:190-194
  fe m = fe_modulus(); fe r; u256_sub(r.l, m.l, a.l);
  bool z = fe_is_zero(a);
#pragma unroll
  for (int i = 0; i < 8; i++) r.l[i] = z ? 0u : r.l[i];
  return r;
}

// ---- 8x8 -> 16 limb product ----------------------------------------------------------------------
// Device: the partial products a_j*b_i are split by the parity of (i+j).  Products of one parity
// never overlap inside a row, so every row is one carry chain of (mad.lo.cc, madc.hi.cc) pairs that
// accumulate a full 32x32+64 result per pair (IMAD.WIDE.U32 with carry in SASS).  e[] collects the
// even columns, o[] the odd ones (o[k] is column k+1); they are merged once at the end.
GW_HD void u256_mul_wide(uint32_t* out, const uint32_t* a, const uint32_t* b) {
#if defined(GW_CHAINS)
  uint32_t e[18], o[18];
#pragma unroll
  for (int i = 0; i < 18; i++) { e[i] = 0; o[i] = 0; }
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const uint32_t bi = b[i];
    const int p = i & 1;
    // same-parity limbs a_j (j = p, p+2, ..): column i+j is even -> e[i+j], e[i+j+1]
    {
      const int c0 = i + p;
      e[c0] = ptx_mad_lo_cc(a[p], bi, e[c0]);
      e[c0 + 1] = ptx_madc_hi_cc(a[p], bi, e[c0 + 1]);
#pragma unroll
      for (int j = p + 2; j < 8; j += 2) {
        e[i + j] = ptx_madc_lo_cc(a[j], bi, e[i + j]);
        e[i + j + 1] = ptx_madc_hi_cc(a[j], bi, e[i + j + 1]);
      }
      e[c0 + 8] = ptx_addc(e[c0 + 8], 0);
    }
    // opposite-parity limbs a_j (j = 1-p, ..): column i+j is odd -> o[i+j-1], o[i+j]
    {
      const int q = 1 - p;
      const int c0 = i + q - 1;
      o[c0] = ptx_mad_lo_cc(a[q], bi, o[c0]);
      o[c0 + 1] = ptx_madc_hi_cc(a[q], bi, o[c0 + 1]);
#pragma unroll
      for (int j = q + 2; j < 8; j += 2) {
        o[i + j - 1] = ptx_madc_lo_cc(a[j], bi, o[i + j - 1]);
        o[i + j] = ptx_madc_hi_cc(a[j], bi, o[i + j]);
      }
      o[c0 + 8] = ptx_addc(o[c0 + 8], 0);
    }
  }
  out[0] = e[0];
  out[1] = ptx_add_cc(e[1], o[0]);
#pragma unroll
  for (int k = 2; k < 15; k++) out[k] = ptx_addc_cc(e[k], o[k - 1]);
  out[15] = ptx_addc(e[15], o[14]);
#else
  uint32_t t[16];
  for (int i = 0; i < 16; i++) t[i] = 0;
  for (int i = 0; i < 8; i++) {
    uint64_t c = 0;
    for (int j = 0; j < 8; j++) { c += (uint64_t)a[j] * b[i] + t[i + j]; t[i + j] = (uint32_t)c; c >>= 32; }
    t[i + 8] = (uint32_t)c;
  }
  for (int i = 0; i < 16; i++) out[i] = t[i];
#endif
}

// a^2 as a 16-limb integer: the 28 cross products a_i*a_j (i < j) accumulated once on the even/odd pair accumulators
// of u256_mul_wide, doubled with funnel shifts, and the 8 diagonal squares added by ONE carry chain of
// (mad.lo.cc, madc.hi.cc) pairs whose addend is the doubled cross sum: 36 wide multiply-accumulates instead of 64.
GW_HD void u256_sqr_wide(uint32_t* out, const uint32_t* a) {
#if defined(GW_CHAINS)
  uint32_t e[16], o[15];
#pragma unroll
  for (int i = 0; i < 16; i++) e[i] = 0;
#pragma unroll
  for (int i = 0; i < 15; i++) o[i] = 0;
#pragma unroll
  for (int i = 0; i < 7; i++) {
    const uint32_t bi = a[i];
    if (i + 2 < 8) {                       // j = i+2, i+4, ..: even columns i+j
      e[2 * i + 2] = ptx_mad_lo_cc(a[i + 2], bi, e[2 * i + 2]);
      e[2 * i + 3] = ptx_madc_hi_cc(a[i + 2], bi, e[2 * i + 3]);
      int jl = i + 2;
#pragma unroll
      for (int j = i + 4; j < 8; j += 2) {
        e[i + j] = ptx_madc_lo_cc(a[j], bi, e[i + j]);
        e[i + j + 1] = ptx_madc_hi_cc(a[j], bi, e[i + j + 1]);
        jl = j;
      }
      if (i + jl + 2 < 16) e[i + jl + 2] = ptx_addc(e[i + jl + 2], 0);
    }
    {                                      // j = i+1, i+3, ..: odd columns i+j, held at o[i+j-1]
      o[2 * i] = ptx_mad_lo_cc(a[i + 1], bi, o[2 * i]);
      o[2 * i + 1] = ptx_madc_hi_cc(a[i + 1], bi, o[2 * i + 1]);
      int jl = i + 1;
#pragma unroll
      for (int j = i + 3; j < 8; j += 2) {
        o[i + j - 1] = ptx_madc_lo_cc(a[j], bi, o[i + j - 1]);
        o[i + j] = ptx_madc_hi_cc(a[j], bi, o[i + j]);
        jl = j;
      }
      if (i + jl + 1 < 15) o[i + jl + 1] = ptx_addc(o[i + jl + 1], 0);
    }
  }
  // cross sum C (columns 1..15; column 0 and e[0], e[1] are empty)
  uint32_t C[16];
  C[0] = 0;
  C[1] = o[0];
  C[2] = ptx_add_cc(e[2], o[1]);
#pragma unroll
  for (int k = 3; k < 15; k++) C[k] = ptx_addc_cc(e[k], o[k - 1]);
  C[15] = ptx_addc(e[15], o[14]);
  // out = 2 C + sum a_i^2 2^(64 i)
  uint32_t D[16];
  D[0] = 0;
#pragma unroll
  for (int k = 1; k < 16; k++) D[k] = (C[k] << 1) | (C[k - 1] >> 31);
  out[0] = ptx_mad_lo_cc(a[0], a[0], D[0]);
  out[1] = ptx_madc_hi_cc(a[0], a[0], D[1]);
#pragma unroll
  for (int i = 1; i < 8; i++) {
    out[2 * i] = ptx_madc_lo_cc(a[i], a[i], D[2 * i]);
    if (i < 7) out[2 * i + 1] = ptx_madc_hi_cc(a[i], a[i], D[2 * i + 1]);
    else out[2 * i + 1] = ptx_madc_hi(a[i], a[i], D[2 * i + 1]);
  }
#else
  u256_mul_wide(out, a, a);
#endif
}

// low 8 limbs of a*b
GW_HD void u256_mul_lo(uint32_t* out, const uint32_t* a, const uint32_t* b) {
#if defined(GW_CHAINS)
  uint32_t e[10], o[10];
#pragma unroll
  for (int i = 0; i < 10; i++) { e[i] = 0; o[i] = 0; }
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const uint32_t bi = b[i];
    const int p = i & 1;
    {
      const int c0 = i + p;           // even columns c0, c0+2, .. <= 7 (its high word may be column 8: dropped)
      if (c0 < 8) {
        e[c0] = ptx_mad_lo_cc(a[p], bi, e[c0]);
        e[c0 + 1] = ptx_madc_hi_cc(a[p], bi, e[c0 + 1]);
#pragma unroll
        for (int j = p + 2; j < 8; j += 2) {
          if (i + j < 8) {
            e[i + j] = ptx_madc_lo_cc(a[j], bi, e[i + j]);
            e[i + j + 1] = ptx_madc_hi_cc(a[j], bi, e[i + j + 1]);
          }
        }
      }
    }
    {
      const int q = 1 - p;
      const int c0 = i + q - 1;       // o index of the odd column i+q
      if (c0 + 1 < 8) {
        o[c0] = ptx_mad_lo_cc(a[q], bi, o[c0]);
        o[c0 + 1] = ptx_madc_hi_cc(a[q], bi, o[c0 + 1]);
#pragma unroll
        for (int j = q + 2; j < 8; j += 2) {
          if (i + j < 8) {
            o[i + j - 1] = ptx_madc_lo_cc(a[j], bi, o[i + j - 1]);
            o[i + j] = ptx_madc_hi_cc(a[j], bi, o[i + j]);
          }
        }
      }
    }
  }
  out[0] = e[0];
  out[1] = ptx_add_cc(e[1], o[0]);
#pragma unroll
  for (int k = 2; k < 7; k++) out[k] = ptx_addc_cc(e[k], o[k - 1]);
  out[7] = ptx_addc(e[7], o[6]);
#else
  uint32_t t[16];
  u256_mul_wide(t, a, b);
  for (int i = 0; i < 8; i++) out[i] = t[i];
#endif
}

// Upper part of a*b for Barrett's quotient estimate: only partial products a_j*b_i with i+j >= 6
// are accumulated (43 of the 64), so out[8..15] is below the true value by less than 2^-60 of one
// unit of out[8]; out[0..5] are not produced (left 0), out[6..7] are partial.
GW_HD void u256_mul_hi_trunc(uint32_t* out, const uint32_t* a, const uint32_t* b) {
#if defined(GW_CHAINS)
  uint32_t e[18], o[18];
#pragma unroll
  for (int i = 0; i < 18; i++) { e[i] = 0; o[i] = 0; }
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const uint32_t bi = b[i];
    const int p = i & 1;
    {
      // same-parity limbs: first j (>= p, parity p) with i + j >= 6
      int j0 = p;
      while (i + j0 < 6) j0 += 2;
      if (j0 < 8) {
        e[i + j0] = ptx_mad_lo_cc(a[j0], bi, e[i + j0]);
        e[i + j0 + 1] = ptx_madc_hi_cc(a[j0], bi, e[i + j0 + 1]);
#pragma unroll
        for (int j = j0 + 2; j < 8; j += 2) {
          e[i + j] = ptx_madc_lo_cc(a[j], bi, e[i + j]);
          e[i + j + 1] = ptx_madc_hi_cc(a[j], bi, e[i + j + 1]);
        }
        e[i + p + 8] = ptx_addc(e[i + p + 8], 0);
      }
    }
    {
      const int q = 1 - p;
      int j0 = q;
      while (i + j0 < 6) j0 += 2;
      if (j0 < 8) {
        o[i + j0 - 1] = ptx_mad_lo_cc(a[j0], bi, o[i + j0 - 1]);
        o[i + j0] = ptx_madc_hi_cc(a[j0], bi, o[i + j0]);
#pragma unroll
        for (int j = j0 + 2; j < 8; j += 2) {
          o[i + j - 1] = ptx_madc_lo_cc(a[j], bi, o[i + j - 1]);
          o[i + j] = ptx_madc_hi_cc(a[j], bi, o[i + j]);
        }
        o[i + q + 7] = ptx_addc(o[i + q + 7], 0);
      }
    }
  }
#pragma unroll
  for (int k = 0; k < 6; k++) out[k] = 0;
  out[6] = ptx_add_cc(e[6], o[5]);
#pragma unroll
  for (int k = 7; k < 15; k++) out[k] = ptx_addc_cc(e[k], o[k - 1]);
  out[15] = ptx_addc(e[15], o[14]);
#else
  uint32_t t[17];
  for (int i = 0; i < 17; i++) t[i] = 0;
  for (int i = 0; i < 8; i++) {
    uint64_t c = 0;
    int jf = 8;
    for (int j = 0; j < 8; j++) {
      if (i + j < 6) continue;
      if (jf == 8) jf = j;
      c += (uint64_t)a[j] * b[i] + t[i + j]; t[i + j] = (uint32_t)c; c >>= 32;
    }
    if (jf < 8) { c += t[i + 8]; t[i + 8] = (uint32_t)c; if (i + 9 < 17) t[i + 9] += (uint32_t)(c >> 32); }
  }
  for (int i = 0; i < 16; i++) out[i] = t[i];
#endif
}

GW_HD uint32_t funnel_r(uint32_t lo, uint32_t hi, uint32_t s) {   // low 32 bits of (hi:lo) >> s, 0 <= s < 32
#if defined(__CUDA_ARCH__)
  return __funnelshift_r(lo, hi, s);
#else
  return s == 0 ? lo : (lo >> s) | (hi << (32 - s));
#endif
}

// 512-bit product (< 2^508) -> [0, M) by Barrett reduction
GW_HD fe fe_barrett(const uint32_t* P) {
  uint32_t q1[8], mu[8], Q[16], qh[8], m[8], T[8];
#pragma unroll
  for (int k = 0; k < 8; k++) { q1[k] = funnel_r(P[7 + k], P[8 + k], 28); mu[k] = MU_L(k); m[k] = MOD_L(k); }  // P >> 252
  u256_mul_hi_trunc(Q, q1, mu);
#pragma unroll
  for (int k = 0; k < 7; k++) qh[k] = funnel_r(Q[8 + k], Q[9 + k], 1);                                         // Q >> 257
  qh[7] = Q[15] >> 1;
  u256_mul_lo(T, qh, m);
  // Quotient estimate: qh = floor(floor(P/2^252) * mu / 2^257) with mu = floor(2^509/M).  With
  // x = P/M:  qh > x - 2^252/M - P/(2^509) - (truncation < 2^-50) - 1 > x - 0.33 - 0.29 - 1, and qh <= x,
  // so floor(x) - 1 <= qh <= floor(x):  0 <= P - qh*M < 2M and ONE conditional subtraction finishes.
  fe r; u256_sub(r.l, P, T);      // P - qh*M < 2M < 2^256, so the low 256 bits are exact
  fe_cond_sub_m(r);
  return r;
}

GW_HD fe fe_mul(const fe& a, const fe& b) {          // graph.rs:105
  uint32_t P[16];
  u256_mul_wide(P, a.l, b.l);
  return fe_barrett(P);
}
GW_HD fe fe_sqr(const fe& a) {
  uint32_t P[16];
  u256_sqr_wide(P, a.l);
  return fe_barrett(P);
}
// two independent products in one basic block (instruction-level parallelism for the scheduler)
GW_HD void fe_mul2(const fe& a1, const fe& b1, const fe& a2, const fe& b2, fe& r1, fe& r2) {
  uint32_t P1[16], P2[16];
  u256_mul_wide(P1, a1.l, b1.l);
  u256_mul_wide(P2, a2.l, b2.l);
  r1 = fe_barrett(P1);
  r2 = fe_barrett(P2);
}
// out-of-line copy for the long chains (inversion, pow): keeps the interpreter's code size down
GW_HD_NOINLINE fe fe_mul_ni(const fe& a, const fe& b) { return fe_mul(a, b); }

// ---- fused linear combinations (OP_DOT): 512-bit accumulator + ONE Montgomery reduction -----------------
// The accumulator holds a 512-bit non-negative integer P; the plan compiler guarantees P < 2^512 (plan.cpp,
// dot_bound).  Device form: the even/odd pair accumulators of u256_mul_wide (e[k] = column k, o[k] = column k + 1),
// never merged -- products are accumulated in place and the Montgomery reduction consumes e and o directly.
struct dot_acc {
#if defined(GW_CHAINS)
  // E[k] = columns 2k, 2k+1 (the e[] pairs of u256_mul_wide); O[k] = columns 2k+1, 2k+2 (the o[] pairs); K[k] counts
  // lazy carries into column 8 + k: P = E + (O << 32) + (K << 256)
  uint64_t E[8], O[7]; uint32_t K[9];
#else
  uint32_t P[16];
#endif
};
#if defined(GW_CHAINS)
GW_HD uint32_t dot_e(const dot_acc& A, int k) { return (k & 1) ? (uint32_t)(A.E[k >> 1] >> 32) : (uint32_t)A.E[k >> 1]; }   // e[k] = column k
GW_HD uint32_t dot_o(const dot_acc& A, int k) { return k >= 14 ? 0u : (k & 1) ? (uint32_t)(A.O[k >> 1] >> 32) : (uint32_t)A.O[k >> 1]; }   // o[k] = column k + 1
#endif
GW_HD void dot_init(dot_acc& A) {
#if defined(GW_CHAINS)
#pragma unroll
  for (int k = 0; k < 8; k++) A.E[k] = 0;
#pragma unroll
  for (int k = 0; k < 7; k++) A.O[k] = 0;
#pragma unroll
  for (int k = 0; k < 9; k++) A.K[k] = 0;
#else
  for (int k = 0; k < 16; k++) A.P[k] = 0;
#endif
}
GW_HD void dot_load(dot_acc& A, const uint32_t* p16) {   // P <- a 16-limb integer
  dot_init(A);
#if defined(GW_CHAINS)
#pragma unroll
  for (int k = 0; k < 8; k++) A.E[k] = pair64(p16[2 * k], p16[2 * k + 1]);
#else
  for (int k = 0; k < 16; k++) A.P[k] = p16[k];
#endif
}
// P += a * b (8 x 8 limbs): the rows of u256_mul_wide; the carry out of every row chain is counted in K.
GW_HD void dot_mac(dot_acc& A, const uint32_t* a, const uint32_t* b) {
#if defined(GW_CHAINS)
  uint32_t* K = A.K;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const uint32_t bi = b[i];
    const int p = i & 1;
    {
      const int c0 = i + p;                // even: columns c0, c0+2, .. pair up in E
      ptx_mac64_first(A.E[c0 >> 1], a[p], bi);
#pragma unroll
      for (int j = p + 2; j < 8; j += 2) ptx_mac64_next(A.E[(i + j) >> 1], a[j], bi);
      K[c0] = ptx_addc(K[c0], 0);          // carry out of the last pair (columns c0+6, c0+7) -> column c0+8
    }
    {
      const int q = 1 - p;
      const int c0 = i + q - 1;            // even: o index of the odd column i + q
      ptx_mac64_first(A.O[c0 >> 1], a[q], bi);
#pragma unroll
      for (int j = q + 2; j < 8; j += 2) ptx_mac64_next(A.O[(i + j - 1) >> 1], a[j], bi);
      K[c0 + 1] = ptx_addc(K[c0 + 1], 0);  // o[c0+8] is column c0+9
    }
  }
#else
  uint32_t Q[16];
  u256_mul_wide(Q, a, b);
  uint64_t c = 0;
  for (int i = 0; i < 16; i++) { c += (uint64_t)A.P[i] + Q[i]; A.P[i] = (uint32_t)c; c >>= 32; }
#endif
}
// P += v (8 limbs) at limb offset `off` (0 or 8), carry propagated to the top
GW_HD void dot_add256(dot_acc& A, const uint32_t* v, int off) {
#if defined(GW_CHAINS)
  const int h = off >> 1;
  ptx_add64_cc(A.E[h], pair64(v[0], v[1]));
#pragma unroll
  for (int i = 1; i < 4; i++) ptx_addc64_cc(A.E[h + i], pair64(v[2 * i], v[2 * i + 1]));
  A.K[off] = ptx_addc(A.K[off], 0);        // column off + 8 (K[8] = column 16 stays 0: P < 2^512)
#else
  uint32_t* P = A.P;
  uint64_t c = 0;
  for (int i = 0; i < 8; i++) { c += (uint64_t)P[off + i] + v[i]; P[off + i] = (uint32_t)c; c >>= 32; }
  for (int i = off + 8; i < 16; i++) { c += P[i]; P[i] = (uint32_t)c; c >>= 32; }
#endif
}
// t = P * 2^-256 mod M for P < 2^512 with t_before_subtraction = (P + m*M) / 2^256 < 2^(n_cond_sub) * M and < 2^256
// (the plan compiler bounds P term by term, see plan.cpp).  Word-serial Montgomery reduction: 8 rounds of
// m = P[i] * (-M^-1) mod 2^32; P += m * M << 32 i, as two carry chains per round (even / odd limbs of M) whose
// carry-outs are collected lazily in K (columns 8..16 are never read by a later round).  The accumulator is clobbered.
GW_HD fe fe_mont_reduce_core(dot_acc& A) {
  fe r;
#if defined(GW_CHAINS)
  // IMAD.WIDE accumulates into an ALIGNED register pair, so a column may only ever be the low half of a pair in one
  // array: E holds pairs starting at even columns (e[k] = column k), O pairs starting at odd columns (o[k] = column
  // k + 1).  Round i clears column i: its low word t = e[i] + o[i-1] + carry decides m; lo(m*M0) makes the column
  // 0 mod 2^32 (carry out = [t != 0] + the carries of forming t) and is never stored.
  // The array whose pairs START at column i takes hi(m*M0) and m*M2, m*M4, m*M6, the other one m*M1 .. m*M7; chain
  // carry-outs (columns i+8, i+9) are counted in K, which no later round reads.  Nothing is ever re-paired.
  uint32_t* K = A.K;
  uint32_t c = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    uint32_t t;
    if (i == 0) { t = dot_e(A, 0); }
    else { const uint64_t s = (uint64_t)dot_e(A, i) + dot_o(A, i - 1) + c; t = (uint32_t)s; c = (uint32_t)(s >> 32); }
    c += (t != 0u) ? 1u : 0u;
    const uint32_t m = t * MONT_INV32;
    if ((i & 1) == 0) {
      // pairs starting at column i live in E
      ptx_machi64_first(A.E[i >> 1], m, MOD_L(0));
#pragma unroll
      for (int j = 2; j < 8; j += 2) ptx_mac64_next(A.E[(i + j) >> 1], m, MOD_L(j));
      K[i] = ptx_addc(K[i], 0);
      ptx_mac64_first(A.O[i >> 1], m, MOD_L(1));
#pragma unroll
      for (int j = 3; j < 8; j += 2) ptx_mac64_next(A.O[(i + j - 1) >> 1], m, MOD_L(j));
      K[i + 1] = ptx_addc(K[i + 1], 0);
    } else {
      // pairs starting at column i live in O (o[i - 1] = column i)
      ptx_machi64_first(A.O[(i - 1) >> 1], m, MOD_L(0));
#pragma unroll
      for (int j = 2; j < 8; j += 2) ptx_mac64_next(A.O[(i + j - 1) >> 1], m, MOD_L(j));
      K[i] = ptx_addc(K[i], 0);
      ptx_mac64_first(A.E[(i + 1) >> 1], m, MOD_L(1));
#pragma unroll
      for (int j = 3; j < 8; j += 2) ptx_mac64_next(A.E[(i + j) >> 1], m, MOD_L(j));
      K[i + 1] = ptx_addc(K[i + 1], 0);
    }
  }
  // columns 8..15: e + o + K + carry of column 7 (the caller's bound makes the total fit 256 bits)
  K[0] += c;
  r.l[0] = ptx_add_cc(dot_e(A, 8), dot_o(A, 7));
#pragma unroll
  for (int k = 1; k < 7; k++) r.l[k] = ptx_addc_cc(dot_e(A, 8 + k), dot_o(A, 7 + k));
  r.l[7] = ptx_addc(dot_e(A, 15), dot_o(A, 14));
  r.l[0] = ptx_add_cc(r.l[0], K[0]);
#pragma unroll
  for (int k = 1; k < 7; k++) r.l[k] = ptx_addc_cc(r.l[k], K[k]);
  r.l[7] = ptx_addc(r.l[7], K[7]);
#else
  uint32_t* P = A.P;
  uint64_t top = 0;                                    // carries out of column 15
  for (int i = 0; i < 8; i++) {
    const uint32_t m = P[i] * MONT_INV32;
    uint64_t c = 0;
    for (int j = 0; j < 8; j++) { c += (uint64_t)m * MOD_L(j) + P[i + j]; P[i + j] = (uint32_t)c; c >>= 32; }
    for (int k = i + 8; k < 16 && c; k++) { c += P[k]; P[k] = (uint32_t)c; c >>= 32; }
    top += c;
  }
  (void)top;                                           // 0 by the caller's bound
  for (int i = 0; i < 8; i++) r.l[i] = P[8 + i];
#endif
  return r;
}
// r < 2^n * M (n = n_cond_sub in 1..3)  ->  [0, M)
GW_HD void fe_cond_sub_n(fe& r, int n_cond_sub) {
  if (n_cond_sub >= 3) fe_cond_sub_ms<2>(r);
  if (n_cond_sub >= 2) fe_cond_sub_ms<1>(r);
  fe_cond_sub_m(r);
}
GW_HD fe fe_mont_reduce(dot_acc& A, int n_cond_sub) {
  fe r = fe_mont_reduce_core(A);
  fe_cond_sub_n(r, n_cond_sub);
  return r;
}
// one OP_DOT term (isa.h TermKind) accumulated into P; x = register value, c = table constant (pre-scaled)
GW_HD void dot_term(dot_acc& A, uint32_t kind, const fe& x, const fe& c) {
  if (kind == 0) {                                     // T_MAC
    dot_mac(A, x.l, c.l);
  } else if (kind == 1) {                              // T_ADDHI
    dot_add256(A, x.l, 8);
  } else if (kind == 2) {                              // T_SUBHI: + (M - x)
    fe m = fe_modulus(); uint32_t t[8];
    u256_sub(t, m.l, x.l);
    dot_add256(A, t, 8);
  } else {                                             // T_CONST
    dot_add256(A, c.l, 0);
  }
}

// Montgomery product a*b*2^-256 mod M (operands < M), CIOS on 32-bit limbs.
GW_HD fe fe_mont_mul(const fe& a, const fe& b) {
  uint32_t t[10];
  for (int i = 0; i < 10; i++) t[i] = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    uint64_t c = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) { c += (uint64_t)a.l[j] * b.l[i] + t[j]; t[j] = (uint32_t)c; c >>= 32; }
    c += t[8]; t[8] = (uint32_t)c; t[9] = (uint32_t)(c >> 32);
    uint32_t mq = t[0] * MONT_INV32;
    c = ((uint64_t)mq * MOD_L(0) + t[0]) >> 32;
#pragma unroll
    for (int j = 1; j < 8; j++) { c += (uint64_t)mq * MOD_L(j) + t[j]; t[j - 1] = (uint32_t)c; c >>= 32; }
    c += t[8]; t[7] = (uint32_t)c; t[8] = t[9] + (uint32_t)(c >> 32);
  }
  fe r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.l[i] = t[i];
  fe_cond_sub_m(r);
  return r;
}
GW_HD fe fe_to_mont(const fe& a) { fe r2; for (int i = 0; i < 8; i++) r2.l[i] = R2_L(i); return fe_mont_mul(a, r2); }
GW_HD fe fe_from_mont(const fe& a) { return fe_mont_mul(a, fe_small(1)); }

// a^e for a 256-bit exponent held per lane (square and multiply, msb first, 254 bits are enough:
// exponents are canonical field values).  Pow is unimplemented! at run time in the reference
// (graph.rs:141-142); build-time meaning a.pow_mod(b, M) (graph.rs:79).
GW_HD_NOINLINE fe fe_pow(const fe& a, const fe& e) {
  fe r = fe_small(1);
#pragma unroll 1
  for (int i = 253; i >= 0; i--) {
    r = fe_mul_ni(r, r);
    uint32_t w = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) w = (k == (i >> 5)) ? e.l[k] : w;
    fe t = fe_mul_ni(r, a);
    bool bit = (w >> (i & 31)) & 1u;
#pragma unroll
    for (int k = 0; k < 8; k++) r.l[k] = bit ? t.l[k] : r.l[k];
  }
  return r;
}

// a^(M-2): inverse, 0 -> 0 (Div by zero yields 0, graph.rs:109).  The exponent is a compile-time
// constant, so the multiply branch is uniform across the warp.
GW_HD_NOINLINE fe fe_inv_fermat(const fe& a) {
  fe r = fe_small(1);
#pragma unroll 1
  for (int i = 253; i >= 0; i--) {
    r = fe_mul_ni(r, r);
    uint32_t w = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) w = (k == (i >> 5)) ? MM2_L(k) : w;
    if ((w >> (i & 31)) & 1u) r = fe_mul_ni(r, a);
  }
  return r;
}

// ---- integer-domain ops ---------------------------------------------------------------------------
// logical right shift of a 256-bit value by n in [0, 255] with static register indexing
GW_HD fe u256_shr(fe a, uint32_t n) {
  uint32_t ws = n >> 5, bs = n & 31;
  if (ws & 4) {
#pragma unroll
    for (int i = 0; i < 8; i++) a.l[i] = (i + 4 < 8) ? a.l[i + 4] : 0u;
  }
  if (ws & 2) {
#pragma unroll
    for (int i = 0; i < 8; i++) a.l[i] = (i + 2 < 8) ? a.l[i + 2] : 0u;
  }
  if (ws & 1) {
#pragma unroll
    for (int i = 0; i < 8; i++) a.l[i] = (i + 1 < 8) ? a.l[i + 1] : 0u;
  }
  fe r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.l[i] = funnel_r(a.l[i], (i + 1 < 8) ? a.l[i + 1] : 0u, bs);
  return r;
}
// left shift truncated to 256 bits, n in [0, 255]
GW_HD fe u256_shl(fe a, uint32_t n) {
  uint32_t ws = n >> 5, bs = n & 31;
  if (ws & 4) {
#pragma unroll
    for (int i = 7; i >= 0; i--) a.l[i] = (i >= 4) ? a.l[i - 4] : 0u;
  }
  if (ws & 2) {
#pragma unroll
    for (int i = 7; i >= 0; i--) a.l[i] = (i >= 2) ? a.l[i - 2] : 0u;
  }
  if (ws & 1) {
#pragma unroll
    for (int i = 7; i >= 0; i--) a.l[i] = (i >= 1) ? a.l[i - 1] : 0u;
  }
  fe r;
#pragma unroll
  for (int i = 7; i >= 0; i--) {
    uint32_t lo = (i >= 1) ? a.l[i - 1] : 0u;
    r.l[i] = bs == 0 ? a.l[i] : ((a.l[i] << bs) | (lo >> (32 - bs)));
  }
  return r;
}
// shift amount as the reference reads it: b == 0 -> 0, b >= 254 -> 254 (meaning "result is 0"), else b
GW_HD uint32_t shift_amount(const fe& b) {
  uint32_t hi = 0;
#pragma unroll
  for (int i = 1; i < 8; i++) hi |= b.l[i];
  return (hi != 0 || b.l[0] >= 254u) ? 254u : b.l[0];
}
GW_HD fe fe_shr(const fe& a, const fe& b) {          // graph.rs:637-672
  uint32_t n = shift_amount(b);
  fe r = u256_shr(a, n & 255u);
  if (n >= 254u) r = fe_zero();
  return r;
}
// graph.rs:621-635; *overflow is set where the reference panics (result >= M), in which case the
// circom semantics ((a << b) & (2^254 - 1)) mod M are returned.
GW_HD fe fe_shl(const fe& a, const fe& b, bool* overflow) {
  uint32_t n = shift_amount(b);
  fe r = u256_shl(a, n & 255u);
  if (n >= 254u) r = fe_zero();
  *overflow = fe_geq_m(r);
  r.l[7] &= 0x3FFFFFFFu;
  fe_cond_sub_m(r);
  return r;
}
// graph.rs:674-717; which: 0 = and, 1 = or, 2 = xor.  *eq_m is set where the reference panics.
GW_HD fe fe_bitop(const fe& a, const fe& b, int which, bool* eq_m) {
  fe d;
#pragma unroll
  for (int i = 0; i < 8; i++) d.l[i] = which == 0 ? (a.l[i] & b.l[i]) : which == 1 ? (a.l[i] | b.l[i]) : (a.l[i] ^ b.l[i]);
  fe m = fe_modulus();
  *eq_m = u256_eq(d.l, m.l);
  fe_cond_sub_m(d);
  return d;
}
GW_HD fe fe_bnot(const fe& a) {                      // circom: (~a & (2^254 - 1)) mod M  (extension)
  fe d;
#pragma unroll
  for (int i = 0; i < 8; i++) d.l[i] = ~a.l[i];
  d.l[7] &= 0x3FFFFFFFu;
  fe_cond_sub_m(d);
  return d;
}
// circom signed comparison, graph.rs:723-769.  which: 0 = lt, 1 = gt, 2 = leq, 3 = geq
GW_HD bool fe_cmp(const fe& a, const fe& b, int which) {
  uint32_t half[8];
#pragma unroll
  for (int i = 0; i < 8; i++) half[i] = HALF_L(i);
  bool an = u256_lt(half, a.l), bn = u256_lt(half, b.l);
  bool lt = u256_lt(a.l, b.l), gt = u256_lt(b.l, a.l);
  if (an != bn) return (which == 0 || which == 2) ? an : bn;
  return which == 0 ? lt : which == 1 ? gt : which == 2 ? !gt : !lt;
}
// unsigned 256-bit division (b != 0): binary long division, 254 uniform steps (a < 2^254)
GW_HD_NOINLINE void u256_divrem(const fe& a, const fe& b, fe* q, fe* r) {
  fe quo = fe_zero(), rem = fe_zero();
#pragma unroll 1
  for (int i = 253; i >= 0; i--) {
    uint32_t w = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) w = (k == (i >> 5)) ? a.l[k] : w;
    uint32_t bit = (w >> (i & 31)) & 1u;
#pragma unroll
    for (int k = 7; k >= 1; k--) rem.l[k] = (rem.l[k] << 1) | (rem.l[k - 1] >> 31);
    rem.l[0] = (rem.l[0] << 1) | bit;
    uint32_t t[8];
    uint32_t borrow = u256_sub(t, rem.l, b.l);
#pragma unroll
    for (int k = 0; k < 8; k++) rem.l[k] = borrow ? rem.l[k] : t[k];
    uint32_t qb = (borrow ? 0u : 1u) << (i & 31);
#pragma unroll
    for (int k = 0; k < 8; k++) quo.l[k] |= (k == (i >> 5)) ? qb : 0u;
  }
  *q = quo; *r = rem;
}

}  // namespace gw
