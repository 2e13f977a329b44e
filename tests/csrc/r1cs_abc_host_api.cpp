// Host build of the per-constraint ABC step of the ABC kernel (csrc/r1cs_eval.cuh: r1cs_abc, r1cs_wire_reduce) over
// the library's compiled program, so that pytest can check it without a GPU.  Built once with the plain host arithmetic
// and once with -DGW_EMULATE_PTX (the device formulations of field.cuh).
#include <string.h>

#include "../../circom-witnesscalc_b200/csrc/r1cs.hpp"
#include "../../circom-witnesscalc_b200/csrc/r1cs_eval.cuh"

using namespace gw;

struct HostAbc { R1csHeader hdr; R1csProgram prog; std::vector<size_t> start; };   // start[k]: first item of constraint k

extern "C" {

void* r1cs_abc_host_load(const uint8_t* data, size_t len) {
  try {
    HostAbc* h = new HostAbc();
    try { parse_r1cs(data, len, h->hdr, h->prog); } catch (...) { delete h; throw; }
    for (size_t pc = 0; pc < h->prog.code.size() / 2;) {
      h->start.push_back(pc);
      pc += 2 + (size_t)h->prog.code[2 * pc] + h->prog.code[2 * pc + 1] + h->prog.code[2 * pc + 2];
    }
    return h;
  } catch (...) {
    return nullptr;
  }
}

void r1cs_abc_host_free(void* h) { delete (HostAbc*)h; }

// constraint k of one witness row (n_wires x 8 limbs): A, B, C (8 limbs each); returns 1 when a wire value it read was
// >= M (and was reduced), else 0
int r1cs_abc_host_eval(void* hp, uint32_t k, const uint32_t* row, uint32_t* abc) {
  const HostAbc& h = *(HostAbc*)hp;
  size_t pc = h.start[k];
  auto next = [&](uint32_t& a, uint32_t& b) { a = h.prog.code[2 * pc]; b = h.prog.code[2 * pc + 1]; pc++; };
  auto wire_val = [&](uint32_t i) { fe r; memcpy(r.l, row + 8 * (size_t)i, 32); return r; };
  auto const_val = [&](uint32_t c) { fe r; memcpy(r.l, h.prog.consts[c].l, 32); return r; };
  bool reduced = false;
  r1cs_abc(next, wire_val, const_val, &reduced, [&](int which, const fe& v) { memcpy(abc + 8 * which, v.l, 32); });
  return reduced ? 1 : 0;
}

}  // extern "C"
