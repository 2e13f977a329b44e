// Evaluation of a compiled R1CS program (r1cs.hpp) for one witness row: the device kernel (r1cs.cu) and the host
// test build (tests/csrc/r1cs_host_api.cpp) run this same code.
#pragma once
#include "field.cuh"
#include "isa.h"

namespace gw {

// <lc, w> mod M for one compiled linear combination of n terms.  next(wire, meta) yields the next term, wire_val(i)
// the witness value of wire i, const_val(j) table constant j.  A value >= M sets *noncanonical (the chunk bound of
// r1cs.cpp holds for values < M only; such a row fails the constraint that reads it).
template <class Next, class WireVal, class ConstVal>
GW_HD fe r1cs_lc(uint32_t n, Next&& next, WireVal&& wire_val, ConstVal&& const_val, bool* noncanonical) {
  fe S = fe_zero();
  dot_acc P;
  dot_init(P);
#pragma unroll 1
  for (uint32_t t = 0; t < n; t++) {
    uint32_t wire, meta;
    next(wire, meta);
    const fe x = wire_val(wire);
    if (x.l[7] >= MOD_L(7) && fe_geq_m(x)) *noncanonical = true;
    const uint32_t kind = meta & 3u;
    if (kind == T_MAC) {
      const fe c = const_val(meta >> 4);
      dot_mac(P, x.l, c.l);
    } else {
      dot_term(P, kind, x, x);                 // T_ADDHI / T_SUBHI
    }
    const uint32_t ncs = (meta >> 2) & 3u;
    if (ncs) {                                 // last term of a chunk
      S = fe_add(S, fe_mont_reduce(P, (int)ncs));
      dot_init(P);
    }
  }
  return S;
}

// a * b == c for canonical a, b, c
GW_HD bool r1cs_holds(const fe& a, const fe& b, const fe& c) {
  uint32_t P[16];
  u256_mul_wide(P, a.l, b.l);
  const fe ab = fe_barrett(P);
  return u256_eq(ab.l, c.l);
}

// A witness value as the ABC evaluation reads it: reduced mod M (like Fr::new on graph inputs), so that <A_k,w>,
// <B_k,w> and <C_k,w> are defined for every row.  *reduced is set when x was >= M: the check's verdict still fails the
// constraint that reads it.
GW_HD fe r1cs_wire_reduce(fe x, bool* reduced) {
  if (x.l[7] >= MOD_L(7) && fe_geq_m(x)) {
    *reduced = true;
    x = fe_reduce256(x);
  }
  return x;
}

// <A_k,w>, <B_k,w>, <C_k,w> of one constraint (its header and terms come from next): emit(which, value) receives each
// value, canonical, as soon as it is reduced (which = 0, 1, 2 for A, B, C).  Wire values >= M are reduced
// (r1cs_wire_reduce) and set *reduced.
template <class Next, class WireVal, class ConstVal, class Emit>
GW_HD void r1cs_abc(Next&& next, WireVal&& wire_val, ConstVal&& const_val, bool* reduced, Emit&& emit) {
  uint32_t na, nb, nc, unused;
  next(na, nb);
  next(nc, unused);
  auto wire = [&](uint32_t i) { return r1cs_wire_reduce(wire_val(i), reduced); };
  bool never = false;                          // reduced values are < M: r1cs_lc never sets it
#pragma unroll 1
  for (int which = 0; which < 3; which++)      // one copy of the term loop for A, B and C
    emit(which, r1cs_lc(which == 0 ? na : which == 1 ? nb : nc, next, wire, const_val, &never));
}

}  // namespace gw
