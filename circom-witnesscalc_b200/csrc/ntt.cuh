// NTT arithmetic over the BN254 scalar field: the butterflies and the twiddle tables.  The device kernels (ntt.cu) and
// the host test build (tests/csrc/ntt_host_api.cpp) compile this same code.
//
// Every value stays canonical ([0, M)); there is no lazy range.  A twiddle is stored pre-scaled, w * 2^256 mod M (the
// OP_DOT / R1CS-constant convention), so one Montgomery reduction of x * (w * 2^256) gives x * w: for x, w' < M the
// product is < M^2 and (M^2 + (2^256 - 1) * M) / 2^256 < 2M, so one conditional subtraction makes it canonical.
#pragma once
#include <vector>

#include "field.cuh"
#include "ntt.hpp"

namespace gw {

// w_28 = 5^((M - 1) / 2^28): 5 is the smallest quadratic non-residue (ffjavascript Fr.w[28], rapidsnark FFT)
GW_HD fe ntt_root28() {
  const uint32_t w[8] = {0x725b19f0u, 0x9bd61b6eu, 0x41112ed4u, 0x402d111eu, 0x8ef62abcu, 0x00e0a7ebu, 0xa58a7e85u, 0x2a3c09f0u};
  fe r;
  for (int i = 0; i < 8; i++) r.l[i] = w[i];
  return r;
}

// x * w mod M for canonical x and a pre-scaled canonical w' = w * 2^256 mod M (bound: see the file comment)
GW_HD fe ntt_mul(const fe& x, const fe& w) {
  dot_acc P;
  dot_init(P);
  dot_mac(P, x.l, w.l);
  return fe_mont_reduce(P, 1);
}

// Gentleman-Sande (decimation in frequency): (a, b) -> (a + b, (a - b) w)
GW_HD void ntt_bfly_dif(fe& a, fe& b, const fe& w) {
  const fe d = fe_sub(a, b);
  a = fe_add(a, b);
  b = ntt_mul(d, w);
}
// Cooley-Tukey (decimation in time): (a, b) -> (a + b w, a - b w)
GW_HD void ntt_bfly_dit(fe& a, fe& b, const fe& w) {
  const fe t = ntt_mul(b, w);
  b = fe_sub(a, t);
  a = fe_add(a, t);
}

// Twiddle tables of one domain n = 2^k, each NTT_TAB pre-scaled entries; a power r^e with e < 2^24 is
// LO[e mod 4096] * HI[e / 4096].  w = w_n, g = w_2n (the coset generator).
static const uint32_t NTT_TAB = 4096;
enum NttTable : uint32_t {
  TW_LO,      // w^t
  TW_HI,      // w^(4096 t)
  ITW_LO,     // w^-t
  ITW_HI,     // w^(-4096 t)
  CG_LO,      // g^t                 forward coset: input i times g^i
  CG_HI,      // g^(4096 t)
  ICG_LO,     // n^-1 g^-t           inverse coset: output i times n^-1 g^-i
  ICG_HI,     // g^(-4096 t)
  QG_LO,      // n^-1 g^t            quotient: inverse output i of B and C times n^-1 g^i (with CG_HI)
  QGR_LO,     // n^-1 g^t 2^256      the same for A: A_odd comes out pre-scaled, so A_odd * B_odd is one ntt_mul
  ROOT,       // w_4096^t, t < 2048  the butterflies of every sub-transform of up to 4096 entries
  IROOT,      // w_4096^-t
  NINV,       // entry 0: n^-1       plain inverse
  NTT_NTAB
};

GW_HD fe ntt_prescale(const fe& x) { fe r1; for (int i = 0; i < 8; i++) r1.l[i] = R1_L(i); return fe_mul(x, r1); }
GW_HD fe ntt_pow2k(fe x, uint32_t k) { for (uint32_t i = 0; i < k; i++) x = fe_mul(x, x); return x; }   // x^(2^k)

// the NTT_NTAB x NTT_TAB table of domain 2^log_n (log_n <= 27), entry t of table j at j * NTT_TAB + t
inline std::vector<fe> ntt_build_tables(uint32_t log_n) {
  std::vector<fe> tab((size_t)NTT_NTAB * NTT_TAB, fe_zero());
  const fe w28 = ntt_root28();
  const fe w = ntt_pow2k(w28, 28 - log_n), g = ntt_pow2k(w28, 27 - log_n), w4096 = ntt_pow2k(w28, 16);
  const fe ninv = fe_inv_fermat(fe_small(1u << log_n));
  auto fill = [&](NttTable j, fe start, const fe& step, uint32_t count) {
    for (uint32_t t = 0; t < count; t++) { tab[(size_t)j * NTT_TAB + t] = ntt_prescale(start); start = fe_mul(start, step); }
  };
  const fe one = fe_small(1);
  const fe wi = fe_inv_fermat(w), gi = fe_inv_fermat(g);
  fill(TW_LO, one, w, NTT_TAB);
  fill(TW_HI, one, ntt_pow2k(w, 12), NTT_TAB);
  fill(ITW_LO, one, wi, NTT_TAB);
  fill(ITW_HI, one, ntt_pow2k(wi, 12), NTT_TAB);
  fill(CG_LO, one, g, NTT_TAB);
  fill(CG_HI, one, ntt_pow2k(g, 12), NTT_TAB);
  fill(ICG_LO, ninv, gi, NTT_TAB);
  fill(ICG_HI, one, ntt_pow2k(gi, 12), NTT_TAB);
  fill(QG_LO, ninv, g, NTT_TAB);
  fill(QGR_LO, ntt_prescale(ninv), g, NTT_TAB);
  fill(ROOT, one, w4096, NTT_TAB / 2);
  fill(IROOT, one, fe_inv_fermat(w4096), NTT_TAB / 2);
  fill(NINV, ninv, one, 1);
  return tab;
}

}  // namespace gw
