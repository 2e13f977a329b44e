// iden3 .r1cs (version 1) reader and constraint compiler.  Layout (little-endian):
//   file    := "r1cs" u32(version = 1) u32(n_sections) section*     sections in any order, each type at most once
//   section := u32(type) u64(size) byte{size}
//   type 1  := u32(n8) prime{n8} u32(n_wires) u32(n_pub_out) u32(n_pub_in) u32(n_prv_in) u64(n_labels) u32(m)
//   type 2  := constraint{m};  constraint := lc(A) lc(B) lc(C);  lc := u32(n) { u32(wire) coeff{n8} }{n}
//   type 3  := u64{n_wires}  (wire -> label; only its length is checked)
//   type 4, 5: PLONK custom gates (circom `pragma custom_templates`): rejected
// Coefficients are plain (not Montgomery) little-endian integers; values >= M are reduced mod M.
#include "r1cs.hpp"

#include <string.h>

#include <algorithm>
#include <numeric>
#include <string>

#include "isa.h"
#include "plan.hpp"

namespace gw {

namespace {

struct Reader {
  const uint8_t* p; const uint8_t* end; const char* what;
  void need(size_t n) const {
    if ((size_t)(end - p) < n) throw Error(std::string("r1cs: truncated ") + what);
  }
  uint32_t u32() { need(4); uint32_t v; memcpy(&v, p, 4); p += 4; return v; }
  uint64_t u64() { need(8); uint64_t v; memcpy(&v, p, 8); p += 8; return v; }
  const uint8_t* bytes(size_t n) { need(n); const uint8_t* q = p; p += n; return q; }
};

U256 m_minus_1() { U256 r = BN254_M; r.l[0] -= 1; return r; }

// The chunk bound.  A chunk of a linear combination accumulates P = sum of its terms in 512 bits; fe_mont_reduce
// returns T = (P + m M) / 2^256 with m < 2^256, then n_cond_sub conditional subtractions.  With every witness value
// and every stored constant <= M - 1 (the worst case: all M - 1):
//   T_MAC   adds x * c'          <= (M - 1)^2        < M * 2^256 * 0.18906   (M / 2^256 = 0.18905..)
//   T_ADDHI adds x << 256        <= (M - 1) * 2^256  < M * 2^256
//   T_SUBHI adds (M - x) << 256  <= M * 2^256         (x = 0)
// so T < M * (1 + 0.18906 n_mac + n_hi).  In thousandths of M: weight = 1000 + 190 n_mac + 1000 n_hi.  A chunk is
// closed before its weight would pass 5250 (< 2^256 / M = 5.2897), which keeps T < 2^256 and P < 2^512:
// at most 22 T_MAC terms, or 4 T_ADDHI/T_SUBHI terms, per reduction.  T < 2^n M for n = 1, 2, 3 when the weight is
// <= 2000, 4000, 5250: that many conditional subtractions give the chunk's value in [0, M).
void close_chunk(R1csProgram& prog, size_t last_item, uint32_t weight) {
  prog.code[2 * last_item + 1] |= r1cs_cond_subs(weight) << 2;
  prog.n_chunks++;
}

// compiles lc into terms appended to prog (zero coefficients are dropped); returns the number of terms emitted
uint32_t compile_lc(const std::vector<std::pair<uint32_t, U256>>& lc, R1csProgram& prog, std::map<U256, uint32_t>& const_index,
                    std::vector<uint64_t>& const_uses) {
  static const U256 zero = U256(), one = u256_from_u64(1), mm1 = m_minus_1();
  uint32_t n = 0, weight = R1CS_W_BASE;
  size_t last = 0;
  for (const auto& t : lc) {
    if (t.second == zero) continue;
    uint32_t kind, cidx = 0, w;
    if (t.second == one) { kind = T_ADDHI; w = R1CS_W_HI; }
    else if (t.second == mm1) { kind = T_SUBHI; w = R1CS_W_HI; }
    else {
      kind = T_MAC; w = R1CS_W_MAC;
      const U256 c = prescale(t.second, false);
      auto it = const_index.find(c);
      if (it == const_index.end()) {
        if (const_uses.size() >= (1u << 28)) throw Error("r1cs: more than 2^28 distinct coefficients");
        it = const_index.emplace(c, (uint32_t)const_uses.size()).first;
        const_uses.push_back(0);
        prog.consts.push_back(c);
      }
      cidx = it->second;
      const_uses[cidx]++;
      prog.n_mac_terms++;
    }
    if (n > 0 && weight + w > R1CS_W_MAX) { close_chunk(prog, last, weight); weight = R1CS_W_BASE; }
    last = prog.code.size() / 2;
    prog.code.push_back(t.first);
    prog.code.push_back(kind | (cidx << 4));
    weight += w;
    n++;
  }
  if (n > 0) close_chunk(prog, last, weight);
  prog.n_terms += n;
  return n;
}

}  // namespace

void parse_r1cs(const uint8_t* data, size_t len, R1csHeader& hdr, R1csProgram& prog) {
  if (!data) throw Error("r1cs: no data");
  Reader f{data, data + len, "file header"};
  if (len < 4 || memcmp(f.bytes(4), "r1cs", 4) != 0) throw Error("r1cs: bad magic (not an .r1cs file)");
  const uint32_t version = f.u32();
  if (version != 1) throw Error("r1cs: unsupported version " + std::to_string(version) + " (only version 1 is known)");
  const uint32_t n_sections = f.u32();
  Reader sec[6] = {};
  bool have[6] = {false, false, false, false, false, false};
  for (uint32_t s = 0; s < n_sections; s++) {
    f.what = "section table";
    const uint32_t type = f.u32();
    const uint64_t size = f.u64();
    if (size > (uint64_t)(f.end - f.p)) throw Error("r1cs: truncated file: section " + std::to_string(type) + " claims " + std::to_string(size) + " bytes");
    const uint8_t* body = f.bytes((size_t)size);
    if (type == 4 || type == 5) throw Error("r1cs: custom gates (section " + std::to_string(type) + ") are not supported");
    if (type >= 1 && type <= 3) {
      if (have[type]) throw Error("r1cs: section " + std::to_string(type) + " appears twice");
      have[type] = true;
      sec[type] = Reader{body, body + size, type == 1 ? "header section" : type == 2 ? "constraints section" : "wire2label section"};
    }
  }
  if (f.p != f.end) throw Error("r1cs: " + std::to_string(f.end - f.p) + " bytes after the last section");
  if (!have[1]) throw Error("r1cs: header section (1) missing");
  if (!have[2]) throw Error("r1cs: constraints section (2) missing");

  Reader& h = sec[1];
  hdr.n8 = h.u32();
  if (hdr.n8 != 32) throw Error("r1cs: field element size n8 = " + std::to_string(hdr.n8) + ": this library evaluates BN254 graphs only (n8 = 32)");
  if (memcmp(h.bytes(32), BN254_M.l, 32) != 0) throw Error("r1cs: the prime is not BN254's: this library evaluates BN254 graphs only");
  hdr.n_wires = h.u32(); hdr.n_pub_out = h.u32(); hdr.n_pub_in = h.u32(); hdr.n_prv_in = h.u32();
  hdr.n_labels = h.u64(); hdr.n_constraints = h.u32();
  if (h.p != h.end) throw Error("r1cs: header section is longer than its content");
  if (have[3] && (uint64_t)(sec[3].end - sec[3].p) != 8ull * hdr.n_wires)
    throw Error("r1cs: wire2label section has " + std::to_string(sec[3].end - sec[3].p) + " bytes, expected 8 x n_wires");

  Reader& c = sec[2];
  // every constraint needs at least 12 bytes: a count that cannot fit is rejected before anything is reserved
  if (hdr.n_constraints > (uint64_t)(c.end - c.p) / 12) throw Error("r1cs: truncated constraints section");
  prog = R1csProgram();
  std::map<U256, uint32_t> const_index;
  std::vector<uint64_t> const_uses;
  std::vector<std::pair<uint32_t, U256>> lc;
  for (uint32_t k = 0; k < hdr.n_constraints; k++) {
    const size_t head = prog.code.size();
    prog.code.resize(head + 4, 0u);                 // {n_a, n_b}, {n_c, 0}
    for (int which = 0; which < 3; which++) {
      const uint32_t nt = c.u32();
      if (nt > (uint64_t)(c.end - c.p) / 36) throw Error("r1cs: truncated constraints section");
      lc.clear();
      for (uint32_t t = 0; t < nt; t++) {
        const uint32_t wire = c.u32();
        if (wire >= hdr.n_wires)
          throw Error("r1cs: constraint " + std::to_string(k) + " uses wire " + std::to_string(wire) + " >= n_wires = " + std::to_string(hdr.n_wires));
        lc.emplace_back(wire, u256_from_le_bytes_mod_order(c.bytes(32), 32));
      }
      prog.code[head + which] = compile_lc(lc, prog, const_index, const_uses);
    }
  }
  if (c.p != c.end) throw Error("r1cs: constraints section is longer than its " + std::to_string(hdr.n_constraints) + " constraints");

  // constant table, most used first (those are the ones staged in shared memory)
  std::vector<uint32_t> order(const_uses.size()), rank(const_uses.size());
  std::iota(order.begin(), order.end(), 0u);
  std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return const_uses[a] > const_uses[b]; });
  std::vector<U256> sorted(order.size());
  for (size_t i = 0; i < order.size(); i++) { rank[order[i]] = (uint32_t)i; sorted[i] = prog.consts[order[i]]; }
  prog.consts.swap(sorted);
  for (size_t pc = 0; pc < prog.code.size();) {
    const size_t nt = (size_t)prog.code[pc] + prog.code[pc + 1] + prog.code[pc + 2];
    pc += 4;
    for (size_t t = 0; t < nt; t++, pc += 2) {
      uint32_t& meta = prog.code[pc + 1];
      if ((meta & 3u) == T_MAC) meta = (meta & 0xFu) | (rank[meta >> 4] << 4);
    }
  }
}

}  // namespace gw
