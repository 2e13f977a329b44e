// Host build of the NTT arithmetic (csrc/ntt.cuh: ntt_mul, the butterflies, ntt_build_tables), so that pytest can check
// it without a GPU.  Built once with the plain host arithmetic and once with -DGW_EMULATE_PTX (the device formulations
// of field.cuh).
#include <string.h>

#include "../../circom-witnesscalc_b200/csrc/ntt.cuh"

using namespace gw;

extern "C" {

uint32_t ntt_host_n_tables() { return NTT_NTAB; }

// the NTT_NTAB x 4096 pre-scaled entries of domain 2^log_n, 32 bytes each
void ntt_host_tables(uint32_t log_n, uint8_t* out) {
  const std::vector<fe> t = ntt_build_tables(log_n);
  memcpy(out, t.data(), t.size() * 32);
}

// which = 0: DIF, 1: DIT, 2: ntt_mul(a, w) into a.  ab: a | b (8 limbs each), updated in place; w pre-scaled
void ntt_host_bfly(int which, uint8_t* a, uint8_t* b, const uint8_t* w) {
  fe x, y, t;
  memcpy(x.l, a, 32); memcpy(y.l, b, 32); memcpy(t.l, w, 32);
  if (which == 0) ntt_bfly_dif(x, y, t);
  else if (which == 1) ntt_bfly_dit(x, y, t);
  else x = ntt_mul(x, t);
  memcpy(a, x.l, 32); memcpy(b, y.l, 32);
}

}  // extern "C"
