// Host build of the R1CS reader/compiler (csrc/r1cs.cpp) and of the evaluation the check kernel runs
// (csrc/r1cs_eval.cuh), so that pytest can check rejections, the compiled program and the chunk bound without a GPU.
// Built once with the plain host arithmetic and once with -DGW_EMULATE_PTX (the device formulations of field.cuh).
#include <string.h>

#include "../../circom-witnesscalc_b200/csrc/r1cs.hpp"
#include "../../circom-witnesscalc_b200/csrc/r1cs_eval.cuh"

using namespace gw;

struct HostR1cs { R1csHeader hdr; R1csProgram prog; std::vector<size_t> start; };   // start[k]: first item of constraint k

extern "C" {

void* r1cs_host_load(const uint8_t* data, size_t len, char* err, size_t err_len) {
  try {
    HostR1cs* h = new HostR1cs();
    try { parse_r1cs(data, len, h->hdr, h->prog); } catch (...) { delete h; throw; }
    for (size_t pc = 0; pc < h->prog.code.size() / 2;) {
      h->start.push_back(pc);
      pc += 2 + (size_t)h->prog.code[2 * pc] + h->prog.code[2 * pc + 1] + h->prog.code[2 * pc + 2];
    }
    return h;
  } catch (const std::exception& e) {
    if (err && err_len) { strncpy(err, e.what(), err_len - 1); err[err_len - 1] = 0; }
    return nullptr;
  }
}

void r1cs_host_free(void* h) { delete (HostR1cs*)h; }

// n_wires, n_pub_out, n_pub_in, n_prv_in, n_constraints, n_labels, n_terms, n_mac_terms, n_chunks, n_consts, n_items
void r1cs_host_info(void* hp, uint64_t* out) {
  const HostR1cs& h = *(HostR1cs*)hp;
  const uint64_t v[11] = {h.hdr.n_wires, h.hdr.n_pub_out, h.hdr.n_pub_in, h.hdr.n_prv_in, h.hdr.n_constraints, h.hdr.n_labels,
                          h.prog.n_terms, h.prog.n_mac_terms, h.prog.n_chunks, h.prog.consts.size(), h.prog.code.size() / 2};
  memcpy(out, v, sizeof v);
}

// constraint k of one witness row (n_wires x 8 limbs): the values of A, B, C (8 limbs each) and whether it holds
// (1), fails (0) or reads a value >= M (2)
int r1cs_host_eval(void* hp, uint32_t k, const uint32_t* row, uint32_t* abc) {
  const HostR1cs& h = *(HostR1cs*)hp;
  size_t pc = h.start[k];
  auto next = [&](uint32_t& a, uint32_t& b) { a = h.prog.code[2 * pc]; b = h.prog.code[2 * pc + 1]; pc++; };
  auto wire_val = [&](uint32_t i) { fe r; memcpy(r.l, row + 8 * (size_t)i, 32); return r; };
  auto const_val = [&](uint32_t c) { fe r; memcpy(r.l, h.prog.consts[c].l, 32); return r; };
  uint32_t n[3], unused;
  next(n[0], n[1]);
  next(n[2], unused);
  bool bad = false;
  fe v[3];
  for (int which = 0; which < 3; which++) {
    v[which] = r1cs_lc(n[which], next, wire_val, const_val, &bad);
    memcpy(abc + 8 * which, v[which].l, 32);
  }
  return bad ? 2 : r1cs_holds(v[0], v[1], v[2]) ? 1 : 0;
}

// the per-row verdict of the check kernel: lowest failing constraint or R1CS_OK
uint32_t r1cs_host_check(void* hp, const uint32_t* row) {
  const HostR1cs& h = *(HostR1cs*)hp;
  uint32_t abc[24];
  for (uint32_t k = 0; k < h.hdr.n_constraints; k++)
    if (r1cs_host_eval(hp, k, row, abc) != 1) return k;
  return R1CS_OK;
}

}  // extern "C"
