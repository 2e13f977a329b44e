#include "plan.hpp"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <array>
#include <map>
#include <set>

#include "field.cuh"

namespace gw {

namespace {

inline int n_operands(const Node& nd) { return nd.kind == N_TRES ? 3 : nd.kind == N_DUO ? 2 : nd.kind == N_UNO ? 1 : 0; }
inline uint32_t operand(const Node& nd, int k) { return k == 0 ? nd.a : k == 1 ? nd.b : nd.c; }

std::vector<uint8_t> liveness(const Graph& g) {
  // dead nodes are unobservable: evaluate() is pure (graph.rs:367)
  const size_t N = g.nodes.size();
  std::vector<uint8_t> needed(N, 0);
  for (uint32_t s : g.witness_signals) needed[s] = 1;
  for (size_t i = N; i-- > 0;) {
    if (!needed[i]) continue;
    const Node& nd = g.nodes[i];
    for (int k = 0; k < n_operands(nd); k++) needed[operand(nd, k)] = 1;
  }
  return needed;
}

inline bool op_has_b_host(uint32_t op) { return op < 32 || op == OP_TERN || op == OP_MULADD; }

fe to_fe(const U256& v) { fe r; memcpy(r.l, v.l, 32); return r; }
U256 to_u256(const fe& v) { U256 r; memcpy(r.l, v.l, 32); return r; }

}  // namespace

U256 prescale(const U256& c, bool neg) {
  fe r1; for (int i = 0; i < 8; i++) r1.l[i] = R1_L(i);
  fe v = to_fe(c);
  if (neg) v = fe_neg(v);
  return to_u256(fe_mul(v, r1));
}

namespace {

// ---- Div batching -----------------------------------------------------------------------------------
// dl(n) = number of Div nodes on the longest operand path ending at n (n itself excluded).  Div nodes with
// equal dl are mutually independent.  The graph is re-emitted level by level (file order inside a level:
// still topological), and the Div nodes of a level are replaced, in groups of <= kmax, by
//   nz_i = NZ1(b_i); p_i = nz_1 .. nz_i; t = INV(p_k); inv_i = t_i * p_(i-1), t_(i-1) = t_i * nz_i;
//   r_i = b_i != 0 ? a_i * inv_i : 0                                    (Div semantics graph.rs:109)
Graph rewrite_div_batches(const Graph& g, uint32_t kmax) {
  const size_t N = g.nodes.size();
  std::vector<uint8_t> needed = liveness(g);
  auto is_div = [&](uint32_t i) { return g.nodes[i].kind == N_DUO && g.nodes[i].op == OP_DIV; };
  std::vector<uint32_t> dl(N, 0);
  uint32_t max_l = 0; size_t n_div = 0;
  for (size_t i = 0; i < N; i++) {
    if (!needed[i]) continue;
    const Node& nd = g.nodes[i];
    uint32_t d = 0;
    for (int k = 0; k < n_operands(nd); k++) { uint32_t o = operand(nd, k); d = std::max(d, dl[o] + (is_div(o) ? 1u : 0u)); }
    dl[i] = d; max_l = std::max(max_l, d);
    n_div += is_div((uint32_t)i);
  }
  if (n_div < 2) return g;
  std::vector<std::vector<uint32_t>> plain(max_l + 1), divs(max_l + 1);
  for (size_t i = 0; i < N; i++) if (needed[i]) (is_div((uint32_t)i) ? divs : plain)[dl[i]].push_back((uint32_t)i);

  Graph ng;
  ng.constants = g.constants; ng.inputs = g.inputs; ng.inputs_size = g.inputs_size;
  ng.nodes.reserve(N + 6 * n_div);
  std::vector<uint32_t> map(N, 0xFFFFFFFFu);
  auto push = [&](uint8_t kind, uint8_t op, uint32_t a, uint32_t b, uint32_t c) {
    Node nd; nd.kind = kind; nd.op = op; nd.a = a; nd.b = b; nd.c = c;
    ng.nodes.push_back(nd);
    return (uint32_t)ng.nodes.size() - 1;
  };
  int32_t zero_node = -1;
  auto const_node = [&](uint64_t v) {
    U256 c = u256_from_u64(v);
    uint32_t ci = 0;
    for (; ci < ng.constants.size(); ci++) if (ng.constants[ci] == c) break;
    if (ci == ng.constants.size()) ng.constants.push_back(c);
    return push(N_CONST, 0, ci, 0, 0);
  };
  auto is_const_one = [&](uint32_t old) {
    const Node& nd = g.nodes[old];
    return nd.kind == N_CONST && g.constants[nd.a] == u256_from_u64(1);
  };
  for (uint32_t L = 0; L <= max_l; L++) {
    for (uint32_t i : plain[L]) {
      const Node& nd = g.nodes[i];
      uint32_t a = nd.a, b = nd.b, c = nd.c;
      if (nd.kind >= N_UNO) a = map[nd.a];
      if (nd.kind >= N_DUO) b = map[nd.b];
      if (nd.kind == N_TRES) c = map[nd.c];
      map[i] = push(nd.kind, nd.op, a, b, c);
    }
    const std::vector<uint32_t>& dv = divs[L];
    for (size_t lo = 0; lo < dv.size(); lo += kmax) {
      const size_t k = std::min<size_t>(kmax, dv.size() - lo);
      if (k == 1) { const Node& nd = g.nodes[dv[lo]]; map[dv[lo]] = push(N_DUO, OP_DIV, map[nd.a], map[nd.b], 0); continue; }
      if (zero_node < 0) zero_node = (int32_t)const_node(0);
      std::vector<uint32_t> nz(k), p(k), inv(k);
      for (size_t i = 0; i < k; i++) nz[i] = push(N_UNO, (uint8_t)(OP_NZ1 - OP_NEG), map[g.nodes[dv[lo + i]].b], 0, 0);
      p[0] = nz[0];
      for (size_t i = 1; i < k; i++) p[i] = push(N_DUO, OP_MUL, p[i - 1], nz[i], 0);
      uint32_t t = push(N_UNO, (uint8_t)(OP_INV - OP_NEG), p[k - 1], 0, 0);
      for (size_t i = k - 1; i >= 1; i--) {
        inv[i] = push(N_DUO, OP_MUL, t, p[i - 1], 0);
        t = push(N_DUO, OP_MUL, t, nz[i], 0);
      }
      inv[0] = t;
      for (size_t i = 0; i < k; i++) {
        const Node& nd = g.nodes[dv[lo + i]];
        uint32_t q = is_const_one(nd.a) ? inv[i] : push(N_DUO, OP_MUL, map[nd.a], inv[i], 0);
        map[dv[lo + i]] = push(N_TRES, 0, map[nd.b], q, (uint32_t)zero_node);
      }
    }
  }
  ng.witness_signals.reserve(g.witness_signals.size());
  for (uint32_t s : g.witness_signals) ng.witness_signals.push_back(map[s]);
  return ng;
}

// ---- narrow typing (isa.h: F_NARROW) -------------------------------------------------------------------
// Interval arithmetic over the graph on the SIGNED reading of field elements (x > M/2 means x - M).  Nothing is
// assumed about inputs; ranges enter through constants, comparisons ({0,1}), masks (Band with a small operand)
// and right shifts, and propagate through Add/Sub/Mul/Neg/TernCond as long as they stay inside (-2^62, 2^62).
// narrow[i] = 1: node i is computed by a narrow instruction (all its operands are readable as int64) and only
// limbs 0..1 of its register are valid.  A wide node with a known range is readable by narrow instructions
// only if the range is non-negative (canonical == zero-extended int64); otherwise its range is forgotten.
struct VRange { bool known = false; int64_t lo = 0, hi = 0; };
struct Typing { std::vector<VRange> rng; std::vector<uint8_t> narrow; };
const int64_t NARROW_LIM = (int64_t)1 << 62;

bool signed_small(const U256& c, int64_t* out) {
  bool small = true;
  for (int k = 2; k < 8; k++) small &= c.l[k] == 0;
  uint64_t lo = (uint64_t)c.l[0] | ((uint64_t)c.l[1] << 32);
  if (small && lo < (uint64_t)NARROW_LIM) { *out = (int64_t)lo; return true; }
  // M - c small?
  uint32_t d[8]; uint64_t borrow = 0;
  for (int k = 0; k < 8; k++) { uint64_t t = (uint64_t)BN254_M.l[k] - c.l[k] - borrow; d[k] = (uint32_t)t; borrow = (t >> 32) & 1u; }
  if (borrow) return false;                      // c > M: not canonical
  for (int k = 2; k < 8; k++) if (d[k]) return false;
  lo = (uint64_t)d[0] | ((uint64_t)d[1] << 32);
  if (lo == 0 || lo >= (uint64_t)NARROW_LIM) return false;
  *out = -(int64_t)lo;
  return true;
}
// the int64 form narrow instructions read from the constant table (limbs 0..1; sign-extended above)
U256 narrow_const(int64_t v) {
  U256 r; const uint32_t ext = v < 0 ? 0xFFFFFFFFu : 0u;
  r.l[0] = (uint32_t)(uint64_t)v; r.l[1] = (uint32_t)((uint64_t)v >> 32);
  for (int k = 2; k < 8; k++) r.l[k] = ext;
  return r;
}

Typing infer_types(const Graph& g, const std::vector<uint8_t>& needed, bool enable) {
  const size_t N = g.nodes.size();
  Typing ty; ty.rng.assign(N, VRange()); ty.narrow.assign(N, 0);
  if (!enable) return ty;
  typedef __int128 i128;
  auto fits = [&](i128 lo, i128 hi) { return lo > -(i128)NARROW_LIM && hi < (i128)NARROW_LIM; };
  auto bits_mask = [&](int64_t a, int64_t b) {     // smallest 2^k - 1 >= max(a, b), a, b >= 0
    uint64_t m = (uint64_t)std::max(a, b), r = 0;
    while (r < m) r = (r << 1) | 1u;
    return (int64_t)r;
  };
  for (size_t i = 0; i < N; i++) {
    if (!needed[i]) continue;
    const Node& nd = g.nodes[i];
    VRange r; bool nar = false;
    auto set = [&](i128 lo, i128 hi) { if (fits(lo, hi)) { r.known = true; r.lo = (int64_t)lo; r.hi = (int64_t)hi; } };
    if (nd.kind == N_CONST) {
      int64_t v; if (signed_small(g.constants.at(nd.a), &v)) set(v, v);
    } else if (nd.kind == N_INPUT) {
      if (nd.a == 0) set(1, 1);                  // get_inputs_buffer forces slot 0 to 1 (lib.rs:177-181)
    } else if (nd.kind == N_UNO) {
      const VRange& a = ty.rng[nd.a];
      const uint32_t op = OP_NEG + nd.op;
      if (op == OP_NEG) { if (a.known) { set(-(i128)a.hi, -(i128)a.lo); nar = r.known; } }
      else if (op == OP_NZ1) { if (a.known) { set(std::min<int64_t>(a.lo, 1), std::max<int64_t>(a.hi, 1)); nar = r.known; } }
      else if (op == OP_WIDEN) { if (a.known) set(a.lo, a.hi); }
      else if (op == OP_LNOT) set(0, 1);
    } else if (nd.kind == N_DUO) {
      const VRange& a = ty.rng[nd.a];
      const VRange& b = ty.rng[nd.b];
      const bool both = a.known && b.known;
      const bool both_nn = both && a.lo >= 0 && b.lo >= 0;
      switch (nd.op) {
        case OP_ADD: if (both) { set((i128)a.lo + b.lo, (i128)a.hi + b.hi); nar = r.known; } break;
        case OP_SUB: if (both) { set((i128)a.lo - b.hi, (i128)a.hi - b.lo); nar = r.known; } break;
        case OP_MUL:
          if (both) {
            i128 p[4] = {(i128)a.lo * b.lo, (i128)a.lo * b.hi, (i128)a.hi * b.lo, (i128)a.hi * b.hi};
            set(std::min(std::min(p[0], p[1]), std::min(p[2], p[3])), std::max(std::max(p[0], p[1]), std::max(p[2], p[3])));
            nar = r.known;
          }
          break;
        case OP_EQ: case OP_NEQ: case OP_LT: case OP_GT: case OP_LEQ: case OP_GEQ: case OP_LAND: case OP_LOR:
          set(0, 1); nar = both; break;
        case OP_BAND:
          if (both_nn) { set(0, std::min(a.hi, b.hi)); nar = true; }
          else if (a.known && a.lo >= 0) set(0, a.hi);
          else if (b.known && b.lo >= 0) set(0, b.hi);
          break;
        case OP_BOR: case OP_BXOR:
          if (both_nn) { set(0, bits_mask(a.hi, b.hi)); nar = r.known; }
          break;
        case OP_SHR:
          if (b.known && b.lo == b.hi && b.lo >= 0) {
            const int64_t k = b.lo;
            if (a.known && a.lo >= 0) { set(0, k >= 63 ? 0 : (a.hi >> k)); nar = true; }
            else if (k >= 254) set(0, 0);
            else if (k >= 192) set(0, (int64_t)((((uint64_t)1 << 62) - 1) >> (k - 192)));   // a < 2^254
          } else if (a.known && a.lo >= 0) {
            set(0, a.hi);                        // a right shift never grows; b >= 254 gives 0
            nar = b.known && b.lo >= 0;
          }
          break;
        case OP_SHL:
          if (a.known && a.lo >= 0 && b.known && b.lo == b.hi && b.lo >= 0 && b.lo < 62) { set(0, (i128)a.hi << b.lo); nar = r.known; }
          break;
        default: break;                          // Div, Pow, Idiv, Mod: wide, unknown
      }
    } else if (nd.kind == N_TRES) {
      const VRange& c = ty.rng[nd.a];
      const VRange& x = ty.rng[nd.b];
      const VRange& y = ty.rng[nd.c];
      if (x.known && y.known) { set(std::min(x.lo, y.lo), std::max(x.hi, y.hi)); nar = c.known && r.known; }
    }
    if (nd.kind >= N_UNO && !nar && r.known && r.lo < 0) r.known = false;
    ty.rng[i] = r;
    ty.narrow[i] = nar ? 1 : 0;
  }
  return ty;
}

// A narrow node read by a wide node goes through one OP_WIDEN node (shared by all its wide consumers).  Dead
// nodes are dropped.  The typing of the new graph is carried over (it is what infer_types would compute).
Graph rewrite_widen(const Graph& g, const std::vector<uint8_t>& needed, const Typing& ty, Typing* ty2) {
  const size_t N = g.nodes.size();
  Graph ng;
  ng.constants = g.constants; ng.inputs = g.inputs; ng.inputs_size = g.inputs_size;
  ng.nodes.reserve(N + N / 8);
  ty2->rng.clear(); ty2->narrow.clear();
  std::vector<uint32_t> map(N, 0xFFFFFFFFu), widened(N, 0xFFFFFFFFu);
  auto push = [&](const Node& nd, const VRange& r, uint8_t nar) {
    ng.nodes.push_back(nd); ty2->rng.push_back(r); ty2->narrow.push_back(nar);
    return (uint32_t)ng.nodes.size() - 1;
  };
  for (size_t i = 0; i < N; i++) {
    if (!needed[i]) continue;
    Node nd = g.nodes[i];
    uint32_t* ops[3] = {&nd.a, &nd.b, &nd.c};
    for (int k = 0; k < n_operands(nd); k++) {
      const uint32_t o = *ops[k];
      if (!ty.narrow[i] && ty.narrow[o]) {
        if (widened[o] == 0xFFFFFFFFu) {
          Node w; w.kind = N_UNO; w.op = (uint8_t)(OP_WIDEN - OP_NEG); w.a = map[o]; w.b = w.c = 0;
          VRange r = ty.rng[o]; if (r.lo < 0) r.known = false;
          widened[o] = push(w, r, 0);
        }
        *ops[k] = widened[o];
      } else {
        *ops[k] = map[o];
      }
    }
    map[i] = push(nd, ty.rng[i], ty.narrow[i]);
  }
  ng.witness_signals.reserve(g.witness_signals.size());
  for (uint32_t s : g.witness_signals) ng.witness_signals.push_back(map[s]);
  return ng;
}

// ---- macro ops -----------------------------------------------------------------------------------------
struct PTerm { uint8_t kind; bool neg; uint32_t node; U256 c; };   // kind: 0 value*const, 1 value, 2 const
struct MOp {
  uint32_t node = 0;              // graph node whose value this op defines
  uint32_t opc = OP_NOP;
  uint32_t in[3] = {0, 0, 0}; int n_in = 0;   // operand nodes of a regular op (constants included)
  std::vector<PTerm> terms;       // OP_DOT
  uint32_t ncs = 1;
  uint32_t shift = 0; U256 mask = U256();  // OP_SHRAND
  bool narrow = false;            // F_NARROW: int64 operands and result
  uint32_t pos2 = NO_POS, pos4 = NO_POS;   // OP_POW5: witness positions of a^2 and a^4
};

// bound of the Montgomery-reduced sum before the conditional subtractions, in units of M:
// (P + mM) / 2^256 < M * (1 + nmac * M / 2^256 + nhi) (+ < 1 for constant terms)
double dot_bound(const std::vector<PTerm>& t) {
  double b = 1.0 + 1e-6;
  for (const PTerm& x : t) b += x.kind == 0 ? 0.18906 : x.kind == 1 ? 1.0 : 1e-9;
  return b;
}

struct Allocator {
  const std::vector<uint32_t>& use_start;
  const std::vector<uint32_t>& use_list;
  std::vector<uint32_t> use_ptr;           // per value: index of its next unconsumed use
  std::vector<int32_t> reg_of, spill_of;   // per value
  std::vector<int32_t> reg_val;            // per register: value or -1
  std::vector<uint32_t> free_regs, free_spill, free_spill_n;   // wide and narrow values spill to separate slot pools
  uint32_t n_spill = 0, n_spill_n = 0;
  Plan& plan;
  const std::vector<uint8_t>* val_narrow = nullptr;    // per value: narrow (8-byte spill moves)
  uint32_t nflag(uint32_t v) const { return (val_narrow && (*val_narrow)[v]) ? (uint32_t)F_NARROW : 0u; }

  Allocator(size_t n, uint32_t n_regs, const std::vector<uint32_t>& us, const std::vector<uint32_t>& ul, Plan& p)
      : use_start(us), use_list(ul), use_ptr(n), reg_of(n, -1), spill_of(n, -1), reg_val(n_regs, -1), plan(p) {
    for (size_t i = 0; i < n; i++) use_ptr[i] = use_start[i];
    for (uint32_t r = n_regs; r-- > 0;) free_regs.push_back(r);
  }
  uint32_t next_use(uint32_t v) const { return use_ptr[v] < use_start[v + 1] ? use_list[use_ptr[v]] : 0xFFFFFFFFu; }
  bool has_uses(uint32_t v) const { return use_ptr[v] < use_start[v + 1]; }
  void emit(const Instr& in) {
    plan.code.push_back(in);
    plan.stats.op_count[in.x & 0x3F]++;
    plan.stats.instrs++;
  }
  // a free register; `pin` = registers that must stay resident for the instruction being built
  uint32_t alloc_reg(const std::vector<uint32_t>& pin) {
    if (!free_regs.empty()) { uint32_t r = free_regs.back(); free_regs.pop_back(); return r; }
    int best = -1; uint32_t best_use = 0;
    for (uint32_t r = 0; r < reg_val.size(); r++) {
      if (std::find(pin.begin(), pin.end(), r) != pin.end()) continue;
      uint32_t nu = next_use((uint32_t)reg_val[r]);
      if (best < 0 || nu > best_use) { best = (int)r; best_use = nu; }
    }
    if (best < 0) throw Error("plan: register file too small for one instruction");
    uint32_t v = (uint32_t)reg_val[best];
    if (spill_of[v] < 0) {                 // first eviction of this value: write it out once (SSA: never changes)
      uint32_t s;
      std::vector<uint32_t>& pool = nflag(v) ? free_spill_n : free_spill;
      if (!pool.empty()) { s = pool.back(); pool.pop_back(); }
      else s = nflag(v) ? n_spill_n++ : n_spill++;
      spill_of[v] = (int32_t)s;
      emit(make_instr(OP_SPILL_ST, nflag(v), NO_DST, (uint32_t)best, s, 0));
      plan.stats.spill_st++;
    }
    reg_of[v] = -1;
    reg_val[best] = -1;
    return (uint32_t)best;
  }
  void bind(uint32_t v, uint32_t r) { reg_of[v] = (int32_t)r; reg_val[r] = (int32_t)v; }
  void release(uint32_t v) {               // value is dead
    if (reg_of[v] >= 0) { reg_val[reg_of[v]] = -1; free_regs.push_back((uint32_t)reg_of[v]); reg_of[v] = -1; }
    if (spill_of[v] >= 0) { (nflag(v) ? free_spill_n : free_spill).push_back((uint32_t)spill_of[v]); spill_of[v] = -1; }
  }
};

// what build_macro_program hands to the two back ends
struct MacroProgram {
  Graph g;                               // the rewritten graph the macro ops refer to (node ids = value ids)
  std::vector<uint8_t> needed, is_const;
  std::vector<U256> const_val;           // canonical value of constant nodes
  Typing ty;
  std::vector<uint32_t> out_start, out_list;   // witness positions per node (CSR)
  std::vector<MOp> mops;
};

// Front half of both plan compilers (throughput and latency mode): graph rewrites, typing, constants, witness
// positions and the macro-op list (linear-combination fusion, Shr+Band fusion).
void build_macro_program(const Graph& g0, const PlanOptions& opt, PlanStats& stats, MacroProgram& mp) {
  stats.graph_nodes = g0.nodes.size();
  stats.graph_ops = g0.n_ops();
  {
    std::vector<uint8_t> nd0 = liveness(g0);
    for (size_t i = 0; i < g0.nodes.size(); i++) {
      if (!nd0[i]) continue;
      stats.live_ops += g0.nodes[i].kind >= N_UNO;
      stats.div_nodes += g0.nodes[i].kind == N_DUO && g0.nodes[i].op == OP_DIV;
      stats.mul_nodes += g0.nodes[i].kind == N_DUO && g0.nodes[i].op == OP_MUL;
    }
  }
  Graph rewritten;
  const bool batch = opt.div_batch > 1 && stats.div_nodes >= 2;
  if (batch) rewritten = rewrite_div_batches(g0, opt.div_batch);
  const Graph& g1 = batch ? rewritten : g0;
  // narrow typing; narrow values read by wide nodes get an explicit OP_WIDEN node
  Typing& ty = mp.ty;
  Graph widened;
  bool any_narrow = false;
  {
    const std::vector<uint8_t> nd1 = liveness(g1);
    Typing t1 = infer_types(g1, nd1, opt.narrow);
    for (uint8_t x : t1.narrow) any_narrow |= x != 0;
    if (any_narrow) widened = rewrite_widen(g1, nd1, t1, &ty); else ty = std::move(t1);
  }
  if (any_narrow) mp.g = std::move(widened); else if (batch) mp.g = std::move(rewritten); else mp.g = g0;
  const Graph& g = mp.g;
  const size_t N = g.nodes.size();
  mp.needed = liveness(g);
  const std::vector<uint8_t>& needed = mp.needed;

  // constants: N_CONST nodes, and Input(0) which get_inputs_buffer forces to 1 (lib.rs:177-181).  const_val is the
  // canonical value; table entries are interned on first use (raw for ordinary operands, pre-scaled for OP_DOT).
  std::vector<uint8_t>& is_const = mp.is_const; is_const.assign(N, 0);
  std::vector<U256>& const_val = mp.const_val; const_val.assign(N, U256());
  for (size_t i = 0; i < N; i++) {
    if (!needed[i]) continue;
    const Node& nd = g.nodes[i];
    if (nd.kind == N_CONST) { is_const[i] = 1; const_val[i] = g.constants.at(nd.a); }
    else if (nd.kind == N_INPUT && nd.a == 0) { is_const[i] = 1; const_val[i] = u256_from_u64(1); }
    else if (nd.kind == N_INPUT && nd.a >= g.inputs_size) throw Error("plan: input index out of range");
  }

  // witness positions per node (CSR), use counts and the single consumer of single-use values
  std::vector<uint32_t>& out_start = mp.out_start; out_start.assign(N + 1, 0);
  std::vector<uint32_t>& out_list = mp.out_list; out_list.assign(g.witness_signals.size(), 0);
  for (uint32_t s : g.witness_signals) out_start[s + 1]++;
  for (size_t i = 0; i < N; i++) out_start[i + 1] += out_start[i];
  {
    std::vector<uint32_t> fill(out_start.begin(), out_start.end() - 1);
    for (uint32_t j = 0; j < g.witness_signals.size(); j++) out_list[fill[g.witness_signals[j]]++] = j;
  }
  std::vector<uint32_t> uses(N, 0), consumer(N, 0);
  for (size_t i = 0; i < N; i++) {
    if (!needed[i]) continue;
    const Node& nd = g.nodes[i];
    for (int k = 0; k < n_operands(nd); k++) { uses[operand(nd, k)]++; consumer[operand(nd, k)] = (uint32_t)i; }
  }
  auto n_out = [&](uint32_t i) { return out_start[i + 1] - out_start[i]; };
  auto is_addsub = [&](uint32_t i) { const Node& nd = g.nodes[i]; return nd.kind == N_DUO && (nd.op == OP_ADD || nd.op == OP_SUB); };

  // ---- macro-op list: linear-combination fusion ---------------------------------------------------------
  const uint32_t max_terms = std::max(1u, std::min(std::min(opt.max_terms, DOT_MAX_TERMS), opt.n_regs - 3));
  const double max_bound = 5.25;                       // 2^256 / M = 5.29: the reduced sum must fit 256 bits
  std::vector<MOp>& mops = mp.mops; mops.clear(); mops.reserve(N);
  std::vector<uint8_t> deferred(N, 0), absorbed(N, 0), addc(N, 0);
  std::map<uint32_t, std::vector<PTerm>> dterms;       // term lists of deferred nodes
  // Shr(x, k) with a constant 0 <= k < 254 whose only consumer is Band(., constant): one OP_SHRAND (Num2Bits, BinSum)
  auto small_const = [&](uint32_t o, uint32_t* v) {
    if (!is_const[o]) return false;
    for (int k = 1; k < 8; k++) if (const_val[o].l[k]) return false;
    *v = const_val[o].l[0];
    return *v < 254u;
  };
  auto shr_absorbable = [&](uint32_t s) {
    const Node& nd = g.nodes[s];
    uint32_t k;
    if (!(nd.kind == N_DUO && nd.op == OP_SHR && !is_const[nd.a] && small_const(nd.b, &k))) return false;
    if (uses[s] != 1 || n_out(s) != 0 || !needed[consumer[s]]) return false;
    const Node& c = g.nodes[consumer[s]];
    if (!(c.kind == N_DUO && c.op == OP_BAND) || c.a == c.b) return false;
    if (ty.narrow[s] && !ty.narrow[consumer[s]]) return false;
    return is_const[c.a == s ? c.b : c.a] != 0;
  };
  auto emit_dot = [&](uint32_t node, std::vector<PTerm>& terms) {
    MOp m; m.node = node; m.opc = OP_DOT; m.terms = std::move(terms); m.narrow = ty.narrow[node] != 0;
    double b = m.narrow ? 1.0 : dot_bound(m.terms);
    m.ncs = b <= 2.0 ? 1 : b <= 4.0 ? 2 : 3;
    mops.push_back(std::move(m));
  };
  auto materialize = [&](uint32_t x) {
    auto it = dterms.find(x);
    emit_dot(x, it->second);
    dterms.erase(it);
    deferred[x] = 0;
  };
  for (size_t idx = 0; idx < N; idx++) {
    const uint32_t i = (uint32_t)idx;
    if (!needed[i] || is_const[i]) continue;
    const Node& nd = g.nodes[i];
    if (nd.kind == N_CONST) continue;
    const bool mul_rc = opt.fuse_dot && nd.kind == N_DUO && nd.op == OP_MUL && (is_const[nd.a] != is_const[nd.b]);
    const bool lin = opt.fuse_dot && is_addsub(i) && !(is_const[nd.a] && is_const[nd.b]);
    if (mul_rc || lin) {
      std::vector<PTerm> terms;
      if (mul_rc) {
        const uint32_t x = is_const[nd.a] ? nd.b : nd.a, c = is_const[nd.a] ? nd.a : nd.b;
        if (addc[x] && !ty.narrow[i]) {
          // S * (y +- C) = S*y +- S*C: the product does not wait for the Add (Poseidon: lc += S * (sigma.out + C))
          const Node& xn = g.nodes[x];
          const bool c_first = is_const[xn.a] != 0;
          const uint32_t y = c_first ? xn.b : xn.a, cc = c_first ? xn.a : xn.b;
          const bool sub = xn.op == OP_SUB;
          terms.push_back(PTerm{0, sub && c_first, y, const_val[c]});
          terms.push_back(PTerm{2, sub && !c_first, 0, to_u256(fe_mul(to_fe(const_val[c]), to_fe(const_val[cc])))});
        } else {
          terms.push_back(PTerm{0, false, x, const_val[c]});
        }
      } else {
        for (int pass = 0; pass < 3; pass++) {
          terms.clear();
          for (int k = 0; k < 2; k++) {
            const uint32_t o = operand(nd, k);
            const bool neg = (k == 1 && nd.op == OP_SUB);
            if (is_const[o]) terms.push_back(PTerm{2, neg, 0, const_val[o]});
            else if (deferred[o]) { for (PTerm t : dterms[o]) { t.neg = (t.neg != neg); terms.push_back(t); } }
            else terms.push_back(PTerm{1, neg, o, U256()});
          }
          if (terms.size() <= max_terms && (ty.narrow[i] || dot_bound(terms) <= max_bound)) break;
          // over budget: turn the larger deferred operand into a plain value and retry
          uint32_t victim = 0xFFFFFFFFu; size_t vsz = 0;
          for (int k = 0; k < 2; k++) { uint32_t o = operand(nd, k); if (!is_const[o] && deferred[o] && dterms[o].size() >= vsz) { victim = o; vsz = dterms[o].size(); } }
          if (victim == 0xFFFFFFFFu) break;
          materialize(victim);
        }
        for (int k = 0; k < 2; k++) {                  // inlined operands are consumed
          const uint32_t o = operand(nd, k);
          if (!is_const[o] && deferred[o]) { dterms.erase(o); deferred[o] = 0; }
        }
      }
      bool has_mac = false;
      for (const PTerm& t : terms) has_mac |= (t.kind == 0);
      if (has_mac || ty.narrow[i]) {                   // narrow sums are always one instruction (no reduction to pay for)
        const bool can_defer = uses[i] == 1 && n_out(i) == 0 && is_addsub(consumer[i]) && needed[consumer[i]] &&
                               ty.narrow[consumer[i]] == ty.narrow[i];
        if (can_defer) { deferred[i] = 1; dterms[i] = std::move(terms); }
        else emit_dot(i, terms);
        continue;
      }
      // a plain Add/Sub of two values: regular op below.  value +- constant read by Mul(constant, .): see mul_rc
      if (opt.fold_addc && !ty.narrow[i] && (is_const[nd.a] != is_const[nd.b])) {
        addc[i] = 1;
        const Node& cn = g.nodes[consumer[i]];
        const bool only_mulc = uses[i] == 1 && n_out(i) == 0 && needed[consumer[i]] && !ty.narrow[consumer[i]] && cn.kind == N_DUO &&
                               cn.op == OP_MUL && cn.a != cn.b && is_const[cn.a == i ? cn.b : cn.a];
        if (only_mulc) continue;                       // its only reader folds it: never materialised
      }
    }
    if (opt.fuse_dot && shr_absorbable(i)) { absorbed[i] = 1; continue; }
    if (nd.kind == N_DUO && nd.op == OP_BAND && (absorbed[nd.a] || absorbed[nd.b])) {
      const uint32_t s = absorbed[nd.a] ? nd.a : nd.b, c = absorbed[nd.a] ? nd.b : nd.a;
      MOp m; m.node = i; m.opc = OP_SHRAND; m.n_in = 1; m.in[0] = g.nodes[s].a;
      m.shift = const_val[g.nodes[s].b].l[0]; m.mask = const_val[c];
      m.narrow = ty.narrow[s] && ty.narrow[i];         // a wide SHRAND writes all 8 limbs: fine for narrow readers
      mops.push_back(m);
      continue;
    }
    MOp m; m.node = i; m.narrow = ty.narrow[i] != 0;
    m.n_in = n_operands(nd);
    for (int k = 0; k < m.n_in; k++) { m.in[k] = operand(nd, k); if (deferred[m.in[k]]) materialize(m.in[k]); }
    if (nd.kind == N_INPUT) m.opc = OP_INPUT;
    else if (nd.kind == N_UNO) m.opc = OP_NEG + nd.op;
    else if (nd.kind == N_TRES) m.opc = OP_TERN;
    else m.opc = (nd.op == OP_MUL && nd.a == nd.b && !is_const[nd.a]) ? (uint32_t)OP_SQR : nd.op;
    mops.push_back(m);
  }
  if (!dterms.empty()) throw Error("plan: dangling deferred linear combination");

}

// Poseidon S-box: Sqr(x) -> Sqr(.) -> Mul(., x) with single-reader intermediates becomes ONE OP_POW5: x stays in
// registers, x^2 and x^4 go straight to their witness positions and never enter the register file / slot file.
// Returns the number of fused chains.
uint64_t fuse_pow5(MacroProgram& mp) {
  const size_t N = mp.g.nodes.size();
  const std::vector<uint32_t>& out_start = mp.out_start; const std::vector<uint32_t>& out_list = mp.out_list;
  auto n_out = [&](uint32_t i) { return out_start[i + 1] - out_start[i]; };
  uint64_t n_fused = 0;
  std::vector<uint32_t> readers(N, 0);
  for (const MOp& m : mp.mops) {
    if (m.opc == OP_DOT) { for (const PTerm& t : m.terms) if (t.kind != 2) readers[t.node]++; }
    else for (int k = 0; k < m.n_in; k++) if (!mp.is_const[m.in[k]] && (k == 0 || m.in[k] != m.in[0]) && (k < 2 || m.in[k] != m.in[1])) readers[m.in[k]]++;   // distinct operands
  }
  std::vector<MOp> fused; fused.reserve(mp.mops.size());
  for (size_t q = 0; q < mp.mops.size(); q++) {
    const MOp& a = mp.mops[q];
    if (q + 2 < mp.mops.size() && a.opc == OP_SQR && !a.narrow && !mp.is_const[a.in[0]]) {
      const MOp& b = mp.mops[q + 1]; const MOp& c = mp.mops[q + 2];
      const bool chain = b.opc == OP_SQR && !b.narrow && b.in[0] == a.node && c.opc == OP_MUL && !c.narrow &&
                         ((c.in[0] == b.node && c.in[1] == a.in[0]) || (c.in[1] == b.node && c.in[0] == a.in[0])) &&
                         readers[a.node] == 1 && readers[b.node] == 1 && n_out(a.node) <= 1 && n_out(b.node) <= 1;
      const uint32_t p2 = chain && n_out(a.node) ? out_list[out_start[a.node]] : NO_POS, p4 = chain && n_out(b.node) ? out_list[out_start[b.node]] : NO_POS;
      // the position of a^4 is encoded relative to that of a^2 (circom numbers in2, in4 consecutively)
      if (chain && (p4 == NO_POS || (p2 != NO_POS && p4 >= p2 && p4 - p2 < 0xFFFFu))) {
        MOp f = c; f.opc = OP_POW5; f.n_in = 1; f.in[0] = a.in[0];
        f.pos2 = p2; f.pos4 = p4;
        fused.push_back(f);
        n_fused++;
        q += 2;
        continue;
      }
    }
    fused.push_back(a);
  }
  mp.mops.swap(fused);
  return n_fused;
}

// Latency plans: take one multiplication per Poseidon round off the critical path.  A partial round is
//   x5 = x^5 (one OP_POW5);  y = S*x5 + (older terms);  next S-box input = y
// i.e. four dependent multiplications from S-box input to S-box input.  With t = S*x computed beside x^2 and x^4,
//   y = t * x^4 + (older terms)
// is three: x -> x^2 -> x^4 -> y (x^5 itself is still computed, for the witness and its other readers, but nobody on the
// path waits for it).  Pattern: an OP_DOT whose value is the input of an OP_POW5 and which has exactly one product term on
// the result of another OP_POW5.  The S-box becomes OP_POW4 + Mul, the linear combination an early OP_DOT + OP_MULADD; the
// new values get node ids behind the graph's.  Field arithmetic is exact, so every value is what it was.
uint64_t rewrite_sbox_links(MacroProgram& mp) {
  const size_t N0 = mp.g.nodes.size();
  std::vector<int32_t> pow5_of(N0, -1);
  std::vector<uint8_t> sbox_in(N0, 0), rewritten(N0, 0);
  for (size_t q = 0; q < mp.mops.size(); q++) if (mp.mops[q].opc == OP_POW5) { pow5_of[mp.mops[q].node] = (int32_t)q; sbox_in[mp.mops[q].in[0]] = 1; }
  // which S-boxes get split, and by which linear combination
  std::vector<int32_t> link_of(mp.mops.size(), -1);       // per OP_DOT: index of the product term on an S-box result
  for (size_t q = 0; q < mp.mops.size(); q++) {
    const MOp& d = mp.mops[q];
    if (d.opc != OP_DOT || d.narrow || d.node >= N0 || !sbox_in[d.node]) continue;
    int32_t hit = -1, n_hit = 0;
    for (size_t k = 0; k < d.terms.size(); k++) if (d.terms[k].kind == 0 && d.terms[k].node < N0 && pow5_of[d.terms[k].node] >= 0) { hit = (int32_t)k; n_hit++; }
    if (n_hit != 1 || rewritten[d.terms[(size_t)hit].node]) continue;      // one link per S-box
    rewritten[d.terms[(size_t)hit].node] = 1;
    link_of[q] = hit;
  }
  auto new_node = [&](bool is_const, const U256& cv) {
    const uint32_t id = (uint32_t)mp.g.nodes.size();
    mp.g.nodes.push_back(Node{N_DUO, (uint8_t)OP_MUL, 0, 0, 0});      // a value id only: never evaluated as a graph node
    mp.needed.push_back(1); mp.is_const.push_back(is_const ? 1 : 0); mp.const_val.push_back(cv);
    mp.ty.rng.push_back(VRange()); mp.ty.narrow.push_back(0);
    mp.out_start.push_back(mp.out_start.back());
    return id;
  };
  std::vector<int32_t> dot_of(N0, -1);                    // per node: the OP_DOT that defines it
  for (size_t q = 0; q < mp.mops.size(); q++) if (mp.mops[q].opc == OP_DOT && mp.mops[q].node < N0) dot_of[mp.mops[q].node] = (int32_t)q;
  uint64_t n_expanded = 0;
  std::vector<uint32_t> x4_of(N0, 0), t_of(N0, 0);        // per S-box result: the ids of x^4 and of t = S*x
  std::vector<MOp> out; out.reserve(mp.mops.size() + mp.mops.size() / 4);
  uint64_t n = 0;
  // the product term of each link, needed when its S-box is met (the S-box comes first in the list)
  std::vector<PTerm> term_of(N0);
  for (size_t q = 0; q < mp.mops.size(); q++) if (link_of[q] >= 0) term_of[mp.mops[q].terms[(size_t)link_of[q]].node] = mp.mops[q].terms[(size_t)link_of[q]];
  for (size_t q = 0; q < mp.mops.size(); q++) {
    const MOp& m = mp.mops[q];
    if (m.opc == OP_POW5 && m.node < N0 && rewritten[m.node]) {
      const uint32_t x = m.in[0], n4 = new_node(false, U256()), nt = new_node(false, U256());
      x4_of[m.node] = n4; t_of[m.node] = nt;
      MOp p4; p4.node = n4; p4.opc = OP_POW4; p4.n_in = 1; p4.in[0] = x; p4.pos2 = m.pos2; p4.pos4 = m.pos4;
      out.push_back(p4);
      MOp t; t.node = nt; t.opc = OP_DOT; PTerm pt = term_of[m.node]; pt.node = x; t.terms.push_back(pt); t.ncs = 1;
      out.push_back(t);
      MOp m5; m5.node = m.node; m5.opc = OP_MUL; m5.n_in = 2; m5.in[0] = n4; m5.in[1] = x;
      out.push_back(m5);
      n++;
      continue;
    }
    if (link_of[q] >= 0) {
      const uint32_t v = m.terms[(size_t)link_of[q]].node;
      // The older terms.  One of them may itself be a linear combination that reads the PREVIOUS round's S-box result
      // (circomlib's sparse mix: s_j' = s_j + S'_j * x5): left alone, x5 -> s_j' -> this sum is a three-deep side path
      // that the shortened chain now overtakes.  So such an operand is written out (its terms scaled by the coefficient,
      // equal values merged: sum_j S_j * s_j' = sum_j S_j * s_j + (sum_j S_j S'_j) * x5), and the sum waits for x5 only.
      struct Coef { uint32_t node; fe c; };                  // signed coefficients as field elements; node 0xFFFFFFFF = the constant
      std::vector<Coef> acc;
      auto add_coef = [&](uint32_t node, const fe& c) {
        for (Coef& a : acc) if (a.node == node) { a.c = fe_add(a.c, c); return; }
        acc.push_back(Coef{node, c});
      };
      auto coef_of = [&](const PTerm& t) { const fe c = t.kind == 1 ? fe_small(1) : to_fe(t.c); return t.neg ? fe_neg(c) : c; };
      bool expanded = false;
      for (size_t k = 0; k < m.terms.size(); k++) {
        if ((int32_t)k == link_of[q]) continue;
        const PTerm& t = m.terms[k];
        const MOp* du = (t.kind != 2 && t.node < N0 && dot_of[t.node] >= 0) ? &mp.mops[(size_t)dot_of[t.node]] : nullptr;
        bool reads_sbox = false;
        if (du) for (const PTerm& u : du->terms) reads_sbox |= u.kind == 0 && u.node < N0 && rewritten[u.node];
        if (du && reads_sbox && !du->narrow) {
          const fe c = coef_of(t);
          for (const PTerm& u : du->terms) add_coef(u.kind == 2 ? 0xFFFFFFFFu : u.node, fe_mul(c, coef_of(u)));
          expanded = true;
        } else add_coef(t.kind == 2 ? 0xFFFFFFFFu : t.node, coef_of(t));
      }
      std::vector<PTerm> rest;
      if (!expanded || acc.size() > 8) { for (size_t k = 0; k < m.terms.size(); k++) if ((int32_t)k != link_of[q]) rest.push_back(m.terms[k]); }
      else {
        for (const Coef& a : acc) {
          if (fe_is_zero(a.c)) continue;
          if (a.node == 0xFFFFFFFFu) rest.push_back(PTerm{2, false, 0, to_u256(a.c)});
          else if (u256_eq(a.c.l, fe_small(1).l)) rest.push_back(PTerm{1, false, a.node, U256()});
          else rest.push_back(PTerm{0, false, a.node, to_u256(a.c)});
        }
        n_expanded++;
      }
      uint32_t c_node;
      if (rest.size() == 1 && rest[0].kind == 1 && !rest[0].neg) c_node = rest[0].node;           // a plain value: no early sum needed
      else if (rest.empty()) c_node = new_node(true, u256_from_u64(0));
      else {
        c_node = new_node(false, U256());
        MOp e; e.node = c_node; e.opc = OP_DOT; e.terms = rest;
        const double b = dot_bound(e.terms); e.ncs = b <= 2.0 ? 1 : b <= 4.0 ? 2 : 3;
        out.push_back(e);
      }
      MOp ma; ma.node = m.node; ma.opc = OP_MULADD; ma.n_in = 3; ma.in[0] = t_of[v]; ma.in[1] = x4_of[v]; ma.in[2] = c_node;
      out.push_back(ma);
      continue;
    }
    out.push_back(m);
  }
  mp.mops.swap(out);
  return n;
}

}  // namespace

Plan compile_plan(const Graph& g0, const PlanOptions& opt) {
  if (opt.n_regs < 4 || opt.n_regs > 4096) throw Error("plan: n_regs out of range");
  Plan plan;
  plan.n_regs = opt.n_regs;
  plan.n_inputs = g0.inputs_size;
  plan.n_witness = (uint32_t)g0.witness_signals.size();
  MacroProgram mp;
  build_macro_program(g0, opt, plan.stats, mp);
  const Graph& g = mp.g;
  const size_t N = g.nodes.size();
  const std::vector<uint8_t>& needed = mp.needed;
  const std::vector<uint8_t>& is_const = mp.is_const;
  const std::vector<U256>& const_val = mp.const_val;
  const Typing& ty = mp.ty;
  const std::vector<uint32_t>& out_start = mp.out_start;
  const std::vector<uint32_t>& out_list = mp.out_list;
  auto n_out = [&](uint32_t i) { return out_start[i + 1] - out_start[i]; };
  if (opt.fuse_pow5) plan.stats.pow5 = fuse_pow5(mp);
  const std::vector<MOp>& mops = mp.mops;
  auto nconst_of = [&](const U256& c, bool neg) {       // int64 table form of a small signed constant
    int64_t v = 0;
    if (!signed_small(c, &v)) throw Error("plan: narrow instruction with a wide constant");
    return narrow_const(neg ? -v : v);
  };
  // table entries are interned on first use (raw for ordinary operands, pre-scaled for OP_DOT)
  std::map<U256, uint32_t> cix;
  auto intern = [&](const U256& v) {
    auto it = cix.find(v);
    if (it == cix.end()) { it = cix.emplace(v, (uint32_t)plan.consts.size()).first; plan.consts.push_back(v); }
    return it->second;
  };

  // value operands (non-constant nodes) of a macro op, without duplicates
  auto value_operands = [&](const MOp& m, std::vector<uint32_t>& v) {
    v.clear();
    if (m.opc == OP_DOT) { for (const PTerm& t : m.terms) if (t.kind != 2 && std::find(v.begin(), v.end(), t.node) == v.end()) v.push_back(t.node); }
    else for (int k = 0; k < m.n_in; k++) if (!is_const[m.in[k]] && std::find(v.begin(), v.end(), m.in[k]) == v.end()) v.push_back(m.in[k]);
  };

  std::vector<uint32_t> vops;
  // use lists of values as macro-op positions of their consumers (CSR, ascending)
  std::vector<uint32_t> use_start(N + 1, 0);
  for (const MOp& m : mops) { value_operands(m, vops); for (uint32_t x : vops) use_start[x + 1]++; }
  for (size_t i = 0; i < N; i++) use_start[i + 1] += use_start[i];
  std::vector<uint32_t> use_list(use_start[N]);
  {
    std::vector<uint32_t> fill(use_start.begin(), use_start.end() - 1);
    for (size_t p = 0; p < mops.size(); p++) { value_operands(mops[p], vops); for (uint32_t x : vops) use_list[fill[x]++] = (uint32_t)p; }
  }

  // constants that are witness signals themselves (e.g. witness[0] = Input(0) = 1)
  Allocator al(N, opt.n_regs, use_start, use_list, plan);
  al.val_narrow = &ty.narrow;
  plan.code.reserve(mops.size() + mops.size() / 2);
  for (size_t i = 0; i < N; i++) {
    if (!needed[i] || !is_const[i]) continue;
    for (uint32_t k = out_start[i]; k < out_start[i + 1]; k++) { al.emit(make_instr(OP_OUT, F_A_CONST, NO_DST, intern(const_val[i]), 0, out_list[k])); plan.stats.outs++; }
  }

  uint32_t live = 0;
  std::vector<uint32_t> pinned, uvops;
  struct Enc { uint32_t enc[3]; uint32_t flags; std::vector<Instr> term_slots; };
  for (size_t p = 0; p < mops.size();) {
    const int n_unit = 1;
    const size_t last = p + n_unit - 1;
    // operands of the whole unit resident
    pinned.clear(); uvops.clear();
    for (int u = 0; u < n_unit; u++) { value_operands(mops[p + u], vops); for (uint32_t x : vops) if (std::find(uvops.begin(), uvops.end(), x) == uvops.end()) uvops.push_back(x); }
    for (uint32_t x : uvops) {
      if (al.reg_of[x] < 0) {
        if (al.spill_of[x] < 0) throw Error("plan: operand neither resident nor spilled");
        uint32_t r = al.alloc_reg(pinned);
        al.emit(make_instr(OP_SPILL_LD, al.nflag(x), r, (uint32_t)al.spill_of[x], 0, 0));
        plan.stats.spill_ld++;
        al.bind(x, r);
      }
      pinned.push_back((uint32_t)al.reg_of[x]);
    }
    // operand encodings (before the operands are retired)
    Enc encs[2];
    for (int u = 0; u < n_unit; u++) {
      const MOp& m = mops[p + u];
      Enc& e = encs[u]; e.enc[0] = e.enc[1] = e.enc[2] = 0; e.flags = m.narrow ? (uint32_t)F_NARROW : 0u;
      if (m.narrow) plan.stats.narrow_instrs++;
      if (m.opc == OP_DOT) {
        std::vector<uint32_t> words;
        // terms ordered products, +value, -value, constant (lanes of a warp then walk the same term kinds together)
        std::vector<PTerm> ts = m.terms;
        std::stable_sort(ts.begin(), ts.end(), [](const PTerm& a, const PTerm& b) {
          auto key = [](const PTerm& t) { return t.kind == 0 ? 0 : t.kind == 1 ? (t.neg ? 2 : 1) : 3; };
          return key(a) < key(b);
        });
        for (const PTerm& t : ts) {
          uint32_t kind = t.kind == 0 ? (uint32_t)T_MAC : t.kind == 2 ? (uint32_t)T_CONST : (t.neg ? (uint32_t)T_SUBHI : (uint32_t)T_ADDHI);
          uint32_t reg = t.kind == 2 ? 0u : (uint32_t)al.reg_of[t.node];
          uint32_t ci = t.kind == 1 ? 0u : intern(m.narrow ? nconst_of(t.c, t.neg) : prescale(t.c, t.neg));
          words.push_back(kind | (reg << 16)); words.push_back(ci);
          plan.stats.dot_terms[kind]++;
        }
        if (words.size() & 2) { words.push_back(0); words.push_back(0); }
        for (size_t k = 0; k < words.size(); k += 4) { Instr sl; sl.x = words[k]; sl.y = words[k + 1]; sl.z = words[k + 2]; sl.w = words[k + 3]; e.term_slots.push_back(sl); }
      } else if (m.opc == OP_INPUT) {
        e.enc[0] = g.nodes[m.node].a;
      } else if (m.opc == OP_SHRAND) {
        e.enc[0] = (uint32_t)al.reg_of[m.in[0]];
        e.enc[1] = m.shift | (intern(m.narrow ? nconst_of(m.mask, false) : m.mask) << 8);
      } else {
        for (int k = 0; k < m.n_in; k++) {
          if (is_const[m.in[k]]) { e.enc[k] = intern(m.narrow ? nconst_of(const_val[m.in[k]], false) : const_val[m.in[k]]); e.flags |= (F_A_CONST << k); }
          else e.enc[k] = (uint32_t)al.reg_of[m.in[k]];
        }
      }
    }
    // retire operands: consume the uses of this unit; operands that die give their register back
    for (uint32_t x : uvops) while (al.use_ptr[x] < use_start[x + 1] && use_list[al.use_ptr[x]] <= last) al.use_ptr[x]++;
    for (uint32_t x : uvops) {
      if (al.has_uses(x)) continue;
      if (al.reg_of[x] >= 0 || al.spill_of[x] >= 0) { al.release(x); live--; }
    }
    // destinations (the second one must not evict the first)
    uint32_t dsts[2] = {NO_DST, NO_DST}; bool need_reg[2], has_uses[2], out_inline[2];
    pinned.clear();
    for (int u = 0; u < n_unit; u++) {
      const MOp& m = mops[p + u];
      const uint32_t no = n_out(m.node);
      has_uses[u] = al.has_uses(m.node);
      out_inline[u] = no >= 1 && m.opc != OP_TERN;             // .w is operand c for TernCond
      need_reg[u] = has_uses[u] || no > (out_inline[u] ? 1u : 0u);
      if (need_reg[u]) {
        dsts[u] = al.alloc_reg(pinned); al.bind(m.node, dsts[u]); pinned.push_back(dsts[u]);
        live++; plan.stats.max_live = std::max(plan.stats.max_live, live);
      }
    }
    for (int u = 0; u < n_unit; u++) {
      const MOp& m = mops[p + u];
      Enc& e = encs[u];
      const uint32_t* outs = &out_list[out_start[m.node]];
      if (out_inline[u]) { e.flags |= F_OUT; plan.stats.outs++; }
      if (m.opc == OP_DOT) {
        al.emit(make_instr(OP_DOT, e.flags, dsts[u], (uint32_t)m.terms.size() | (m.ncs << 8), 0, out_inline[u] ? outs[0] : 0));
        for (const Instr& sl : e.term_slots) plan.code.push_back(sl);
      } else if (m.opc == OP_POW5) {
        al.emit(make_instr(OP_POW5, e.flags, dsts[u], e.enc[0] | ((m.pos4 == NO_POS ? 0xFFFFu : m.pos4 - m.pos2) << 16), m.pos2, out_inline[u] ? outs[0] : 0));
        plan.stats.outs += (m.pos2 != NO_POS) + (m.pos4 != NO_POS);
      } else {
        const uint32_t w = m.opc == OP_TERN ? e.enc[2] : (out_inline[u] ? outs[0] : 0);
        al.emit(make_instr(m.opc, e.flags, dsts[u], e.enc[0], e.enc[1], w));
      }
      if (m.opc == OP_DIV || m.opc == OP_INV) plan.stats.inversions++;
    }
    for (int u = 0; u < n_unit; u++) {
      const MOp& m = mops[p + u];
      const uint32_t no = n_out(m.node);
      const uint32_t* outs = &out_list[out_start[m.node]];
      for (uint32_t k = out_inline[u] ? 1u : 0u; k < no; k++) { al.emit(make_instr(OP_OUT, al.nflag(m.node), NO_DST, dsts[u], 0, outs[k])); plan.stats.outs++; }
      if (need_reg[u] && !has_uses[u]) { al.release(m.node); live--; }
    }
    p += n_unit;
  }
  plan.n_spill = al.n_spill;
  plan.n_spill_narrow = al.n_spill_n;
  plan.stats.slots = plan.code.size();
  if (plan.consts.empty()) plan.consts.push_back(u256_from_u64(0));

  // most used constants first: the kernel stages a prefix of the table in shared memory
  {
    auto for_each_const_ref = [&](auto&& fn) {
      for (size_t pc = 0; pc < plan.code.size();) {
        Instr& h = plan.code[pc];
        const uint32_t op = h.x & 0xFFu, len = instr_slots(h);
        if (op == OP_DOT) {
          const uint32_t nt = h.y & 0xFFu;
          for (uint32_t t = 0; t < nt; t++) {
            Instr& sl = plan.code[pc + 1 + (t >> 1)];
            const uint32_t kind = ((t & 1) ? sl.z : sl.x) & 0xFu;
            if (kind == T_MAC || kind == T_CONST) fn((t & 1) ? sl.w : sl.y);
          }
        } else if (op == OP_SHRAND) {
          uint32_t ci = h.z >> 8; fn(ci); h.z = (h.z & 0xFFu) | (ci << 8);
        } else if (op != OP_INPUT && op != OP_SPILL_LD && op != OP_SPILL_ST && op != OP_NOP) {
          if (h.x & F_A_CONST) fn(h.y);
          if ((h.x & F_B_CONST) && op_has_b_host(op)) fn(h.z);
          if ((h.x & F_C_CONST) && op == OP_TERN) fn(h.w);
        }
        pc += len;
      }
    };
    std::vector<uint64_t> cnt(plan.consts.size(), 0);
    for_each_const_ref([&](uint32_t& ci) { cnt[ci]++; });
    std::vector<uint32_t> byuse(plan.consts.size());
    for (uint32_t k = 0; k < byuse.size(); k++) byuse[k] = k;
    std::stable_sort(byuse.begin(), byuse.end(), [&](uint32_t a, uint32_t b) { return cnt[a] > cnt[b]; });
    std::vector<uint32_t> new_ix(plan.consts.size());
    std::vector<U256> sorted(plan.consts.size());
    for (uint32_t k = 0; k < byuse.size(); k++) { new_ix[byuse[k]] = k; sorted[k] = plan.consts[byuse[k]]; }
    plan.consts.swap(sorted);
    for_each_const_ref([&](uint32_t& ci) { ci = new_ix[ci]; });
  }
  return plan;
}

}  // namespace gw

namespace gw {

namespace {

// one instruction of the latency plan before slots are assigned
struct LOp {
  uint32_t opc = OP_NOP;
  uint32_t val = 0xFFFFFFFFu;          // value it defines: a graph node, or N + k for the early part of a split OP_DOT
  uint32_t in[3] = {0, 0, 0}; int n_in = 0;   // operands of a regular op (graph nodes, constants included); OP_OUT: in[0]
  std::vector<PTerm> terms; uint32_t ncs = 1; // OP_DOT
  uint32_t shift = 0; U256 mask = U256();   // OP_SHRAND
  uint32_t input = 0;                  // OP_INPUT
  uint32_t level = 0;
  bool has_out = false; uint32_t out_pos = 0;  // inline witness store (F_OUT), or the position of an OP_OUT
  bool slow = false;
  int32_t chain_prev = -1, chain_next = -1;    // a chain runs in ONE lane, back to back, inside one level
  uint32_t pos2 = NO_POS, pos4 = NO_POS;       // OP_POW5
};

inline bool lat_is_slow(uint32_t opc) { return opc == OP_DIV || opc == OP_INV || opc == OP_POW || opc == OP_IDIV || opc == OP_MOD; }

// cycles of one instruction in one lane of the latency kernel, measured in place on a B200 (profiles/r01n/latency.md):
// the arithmetic (tools/ubench/oplat.cu: Mul 920, Sqr 780, one OP_DOT product 800, inversion 41 750) plus what every
// instruction pays around it -- header and operand fetch from shared memory, dispatch, result and witness stores
uint32_t lat_cost(const LOp& o) {
  const uint32_t around = 450;
  switch (o.opc) {
    case OP_MUL: return 1100 + around;
    case OP_SQR: return 950 + around;
    case OP_POW5: return 950 + 950 + 1100 + around + 100;
    case OP_POW4: return 950 + 950 + around + 100;
    case OP_MULADD: return 1100 + 80 + around;
    case OP_DOT: {
      uint32_t c = 1500;
      for (const PTerm& t : o.terms) c += t.kind == 0 ? 800u : 100u;
      return c;
    }
    case OP_ADD: case OP_SUB: return 80 + 300;
    case OP_DIV: return 42700;
    case OP_INV: return 41750;
    case OP_POW: return 450000;
    case OP_IDIV: case OP_MOD: return 40000;
    default: return 60 + 300;
  }
}
// instructions with the same key run the same code path: they can share the lanes of one warp
uint64_t lat_class(const LOp& o) {
  uint64_t k = o.opc;
  if (o.opc == OP_DOT) {
    uint32_t n[3] = {0, 0, 0};
    for (const PTerm& t : o.terms) n[t.kind]++;
    k |= (uint64_t)n[0] << 8 | (uint64_t)n[1] << 16 | (uint64_t)n[2] << 24;
  }
  return k;
}

const uint32_t LAT_LEVEL_OVERHEAD = 500;   // cycles per level around the instructions: packet fetch, descriptor, barrier

}  // namespace

static LatencyPlan compile_latency_plan_one(const Graph& g0, const LatencyOptions& lo);

// The S-box link rewrite shortens a Poseidon chain that has the SM to itself (Poseidon(1): 0.206 -> 0.177 ms) and costs
// a graph that keeps every warp busy anyway (authV2, three hashes side by side: 17.0 -> 21.4 ms; profiles/r02x): it adds
// two packets per round.  Both plans are built and the timing model, which gets both directions right, picks one.
LatencyPlan compile_latency_plan(const Graph& g0, const LatencyOptions& lo) {
  if (lo.fuse && lo.sbox_links && lo.force_sbox_links) return compile_latency_plan_one(g0, lo);
  LatencyOptions plain = lo;
  plain.sbox_links = false;
  // (dataflow plans only: the level plan's cost model is not calibrated for the choice -- it prefers the rewrite on authV2,
  // where the kernel then measures 19.9 instead of 18.9 ms)
  if (!(lo.fuse && lo.sbox_links && lo.dataflow)) return compile_latency_plan_one(g0, plain);
  LatencyPlan a = compile_latency_plan_one(g0, plain);
  try {
    LatencyPlan b = compile_latency_plan_one(g0, lo);
    if (b.n_sbox_links > 0 && b.est_cycles < a.est_cycles) return b;
  } catch (const Error&) { }       // e.g. the rewritten graph keeps more values alive than the slot file holds
  return a;
}

static LatencyPlan compile_latency_plan_one(const Graph& g0, const LatencyOptions& lo) {
  if (lo.n_warps < 1 || lo.n_warps > 16 || lo.n_slow_warps < 1 || lo.n_slow_warps > 6) throw Error("latency plan: warp counts out of range");
  if (lo.max_slots > 0xFFFFu) throw Error("latency plan: value file too large for 16-bit slot numbers");
  PlanOptions po;
  po.n_regs = 64; po.div_batch = 1; po.narrow = false; po.fuse_dot = lo.fuse; po.fold_addc = lo.fuse; po.max_terms = 8;
  PlanStats pst;
  MacroProgram mp;
  build_macro_program(g0, po, pst, mp);
  if (lo.fuse) fuse_pow5(mp);
  uint64_t n_links = 0;
  if (lo.fuse && lo.sbox_links) n_links = rewrite_sbox_links(mp);
  const Graph& g = mp.g;
  const size_t N = g.nodes.size();
  const std::vector<uint8_t>& is_const = mp.is_const;
  auto n_out = [&](uint32_t i) { return mp.out_start[i + 1] - mp.out_start[i]; };

  bool use_chain = lo.chain;
  const int dbg_level = getenv("GW_LAT_DEBUG") ? atoi(getenv("GW_LAT_DEBUG")) : -1;
  const uint32_t dbg_count = getenv("GW_LAT_DEBUG_N") ? (uint32_t)atoi(getenv("GW_LAT_DEBUG_N")) : 24u;
  auto schedule = [&](const uint32_t D) {
    LatencyPlan lp;
    lp.n_inputs = g0.inputs_size;
    lp.n_witness = (uint32_t)g0.witness_signals.size();
    lp.n_warps = lo.n_warps; lp.n_slow_warps = lo.n_slow_warps; lp.slow_levels = D;
    // ---- 1. instructions and their levels (ASAP; a long op delivers D levels after its issue) -------------
    std::vector<LOp> ops; ops.reserve(mp.mops.size() + mp.mops.size() / 4);
    std::vector<uint32_t> chain_len, chain_head;      // per op: the head of its chain; per head: the chain's length
    std::vector<uint32_t> chain_slots;                // per head: packet slots of the chain (headers + tails + constants)
    auto mop_slots = [&](const MOp& m) {
      uint32_t n = 1;
      if (m.opc == OP_DOT) { n += ((uint32_t)m.terms.size() + 1) / 2; for (const PTerm& t : m.terms) n += t.kind != 1 ? 2u : 0u; }
      else if (m.opc == OP_SHRAND) n += 2;
      else for (int k = 0; k < m.n_in; k++) n += is_const[m.in[k]] ? 2u : 0u;
      return n;
    };
    std::vector<uint32_t> avail(N, 0);               // first level that may read the value
    uint32_t n_levels = 1;
    for (size_t i = 0; i < N; i++) {                 // constants that are witness signals themselves (witness[0] = 1)
      if (!mp.needed[i] || !is_const[i]) continue;
      for (uint32_t k = mp.out_start[i]; k < mp.out_start[i + 1]; k++) {
        LOp o; o.opc = OP_OUT; o.n_in = 1; o.in[0] = (uint32_t)i; o.level = 0; o.has_out = true; o.out_pos = mp.out_list[k];
        chain_len.push_back(1); chain_head.push_back((uint32_t)ops.size()); chain_slots.push_back(8);
        ops.push_back(o);
      }
    }
    // readers per value: macro ops that read it (+ the separate OP_OUT stores).  A value with ONE reader whose other
    // operands are older is chained to it: the reader runs in the same lane right after its producer, inside the same
    // level (program order replaces the barrier), e.g. the x^2, x^4, x^5 of a Poseidon S-box become one level.
    std::vector<uint32_t> n_readers(N, 0);
    {
      std::vector<uint32_t> seen;
      for (const MOp& m : mp.mops) {
        seen.clear();
        auto rd = [&](uint32_t v) { if (std::find(seen.begin(), seen.end(), v) == seen.end()) { seen.push_back(v); n_readers[v]++; } };
        if (m.opc == OP_DOT) { for (const PTerm& t : m.terms) if (t.kind != 2) rd(t.node); }
        else for (int k = 0; k < m.n_in; k++) if (!is_const[m.in[k]]) rd(m.in[k]);
        const uint32_t no = n_out(m.node);
        if (no > ((no >= 1 && m.opc != OP_TERN && m.opc != OP_MULADD) ? 1u : 0u)) n_readers[m.node] += 2;      // separate stores read the slot later
      }
    }
    std::vector<int32_t> def_op(N, -1);
    for (const MOp& m : mp.mops) {
      LOp o; o.opc = m.opc; o.val = m.node; o.n_in = m.n_in; o.shift = m.shift; o.mask = m.mask; o.ncs = m.ncs;
      o.pos2 = m.pos2; o.pos4 = m.pos4;
      for (int k = 0; k < m.n_in; k++) o.in[k] = m.in[k];
      if (m.opc == OP_INPUT) o.input = g.nodes[m.node].a;
      uint32_t lv = 0;
      // chain candidate: the single newest operand, produced one level earlier by an ordinary instruction that nobody else reads
      int32_t chain_to = -1;
      // (only multiplication-class instructions: a chain of cheap ones would serialise what the lanes of a warp run in parallel)
      if (use_chain && (m.opc == OP_MUL || m.opc == OP_SQR || m.opc == OP_DOT || m.opc == OP_POW5)) {
        uint32_t newest = 0xFFFFFFFFu, amax = 0, n_at_max = 0;
        auto look = [&](uint32_t v) { if (avail[v] > amax) { amax = avail[v]; newest = v; n_at_max = 1; } else if (avail[v] == amax && v != newest) n_at_max++; };
        if (m.opc == OP_DOT) { for (const PTerm& t : m.terms) if (t.kind != 2) look(t.node); }
        else for (int k = 0; k < m.n_in; k++) if (!is_const[m.in[k]]) look(m.in[k]);
        if (amax > 0 && n_at_max == 1 && newest < N && def_op[newest] >= 0 && n_readers[newest] == 1) {
          const LOp& pr = ops[(size_t)def_op[newest]];
          bool ok = (pr.opc == OP_MUL || pr.opc == OP_SQR || pr.opc == OP_DOT || pr.opc == OP_POW5) && pr.level + 1 == amax && chain_len[chain_head[(size_t)def_op[newest]]] < lo.max_chain &&
                    1 + chain_slots[chain_head[(size_t)def_op[newest]]] + mop_slots(m) <= lo.packet_slots;     // a chain lives in one packet
          auto older = [&](uint32_t v) { if (v != newest && avail[v] > pr.level) ok = false; };
          if (m.opc == OP_DOT) { for (const PTerm& t : m.terms) if (t.kind != 2) older(t.node); }
          else for (int k = 0; k < m.n_in; k++) if (!is_const[m.in[k]]) older(m.in[k]);
          if (ok) chain_to = def_op[newest];
        }
      }
      if (m.opc == OP_DOT) {
        o.terms = m.terms;
        uint32_t rmax = 0;
        for (const PTerm& t : o.terms) if (t.kind != 2) rmax = std::max(rmax, avail[t.node]);
        if (lo.split_dot && rmax > 0 && chain_to < 0) {
          // operands known before rmax go to an early OP_DOT whose reduced sum enters the late one as a plain value
          std::vector<PTerm> early, late;
          bool early_mac = false;
          for (const PTerm& t : o.terms) {
            const bool e = t.kind == 2 || avail[t.node] < rmax;
            (e ? early : late).push_back(t);
            early_mac |= e && t.kind == 0;
          }
          if (early_mac && !late.empty()) {
            const uint32_t ev = (uint32_t)avail.size();
            late.push_back(PTerm{1, false, ev, U256()});
            if (dot_bound(late) <= 5.25) {
              LOp e; e.opc = OP_DOT; e.val = ev; e.terms = std::move(early);
              const double b = dot_bound(e.terms); e.ncs = b <= 2.0 ? 1 : b <= 4.0 ? 2 : 3;
              uint32_t el = 0;
              for (const PTerm& t : e.terms) if (t.kind != 2) el = std::max(el, avail[t.node]);
              e.level = el;
              avail.push_back(el + 1);
              chain_len.resize(ops.size() + 1, 1); chain_head.resize(ops.size() + 1, 0); chain_slots.resize(ops.size() + 1, 8); chain_head[ops.size()] = (uint32_t)ops.size();
              ops.push_back(std::move(e));
              o.terms = std::move(late);
              const double bl = dot_bound(o.terms); o.ncs = bl <= 2.0 ? 1 : bl <= 4.0 ? 2 : 3;
              lp.n_split++;
            }
          }
        }
        for (const PTerm& t : o.terms) if (t.kind != 2) lv = std::max(lv, avail[t.node]);
      } else {
        for (int k = 0; k < m.n_in; k++) if (!is_const[m.in[k]]) lv = std::max(lv, avail[m.in[k]]);
      }
      if (chain_to >= 0) { lv = ops[(size_t)chain_to].level; o.chain_prev = chain_to; ops[(size_t)chain_to].chain_next = (int32_t)ops.size(); lp.n_chained++; }
      o.level = lv;
      o.slow = lat_is_slow(m.opc);
      avail[m.node] = lv + (o.slow ? D : 1u);
      def_op[m.node] = (int32_t)ops.size();
      chain_len.resize(ops.size() + 1, 1); chain_head.resize(ops.size() + 1, 0); chain_slots.resize(ops.size() + 1, 8);
      if (chain_to >= 0) { chain_head[ops.size()] = chain_head[(size_t)chain_to]; chain_len[chain_head[ops.size()]]++; chain_slots[chain_head[ops.size()]] += mop_slots(m); }
      else { chain_head[ops.size()] = (uint32_t)ops.size(); chain_slots[ops.size()] = mop_slots(m); }
      if (o.slow) { lp.n_slow++; n_levels = std::max(n_levels, lv + D); }
      const uint32_t no = n_out(m.node);
      const bool inline_out = no >= 1 && m.opc != OP_TERN && m.opc != OP_MULADD;     // .w is operand c for TernCond and OP_MULADD
      if (inline_out) { o.has_out = true; o.out_pos = mp.out_list[mp.out_start[m.node]]; }
      n_levels = std::max(n_levels, lv + 1);
      ops.push_back(std::move(o));
      for (uint32_t k = inline_out ? 1u : 0u; k < no; k++) {
        LOp w; w.opc = OP_OUT; w.n_in = 1; w.in[0] = m.node; w.level = avail[m.node]; w.has_out = true;
        w.out_pos = mp.out_list[mp.out_start[m.node] + k];
        n_levels = std::max(n_levels, w.level + 1);
        chain_len.resize(ops.size() + 1, 1); chain_head.resize(ops.size() + 1, 0); chain_slots.resize(ops.size() + 1, 8); chain_head[ops.size()] = (uint32_t)ops.size();
        ops.push_back(w);
      }
    }
    const size_t NV = avail.size();

    // ---- 2. last level that reads each value (a long op may read its operands until the level at which it is waited for) -----
    std::vector<int64_t> last_use(NV, -1);
    auto for_operands = [&](const LOp& o, auto&& fn) {
      if (o.opc == OP_DOT) { for (const PTerm& t : o.terms) if (t.kind != 2) fn(t.node); }
      else for (int k = 0; k < o.n_in; k++) if (o.in[k] >= N || !is_const[o.in[k]]) fn(o.in[k]);
    };
    for (const LOp& o : ops) {
      const int64_t rd = o.slow ? (int64_t)o.level + D - 1 : (int64_t)o.level;
      for_operands(o, [&](uint32_t v) { last_use[v] = std::max(last_use[v], rd); });
    }
    std::vector<std::vector<uint32_t>> by_level(n_levels);
    for (size_t k = 0; k < ops.size(); k++) by_level[ops[k].level].push_back((uint32_t)k);

    // ---- 3. level by level: slots, jobs of the slow warps, warp assignment, headers ------------------------
    std::vector<int32_t> slot_of(NV, -1);
    std::vector<uint32_t> free_slots;
    std::vector<std::vector<uint32_t>> dying(n_levels);
    uint32_t n_slots = 0;
    // A packet is what one warp needs for one level (or one slow-warp job), contiguous: slot 0 = descriptor, then the
    // headers, then what the headers point at with packet-relative slot offsets: OP_DOT tails and every constant
    // (two slots each) -- so one asynchronous copy brings a level's instructions AND their constants on chip.
    std::vector<std::vector<std::array<uint32_t, 2>>> pending_waits(n_levels);
    std::vector<std::vector<std::array<uint32_t, 3>>> jobq(lo.n_slow_warps);
    std::vector<uint64_t> busy(lo.n_slow_warps, 0);
    std::vector<std::array<uint32_t, 4>> pinfo;      // per (physical level, warp): offset, slots, headers, lanes
    uint32_t n_phys = 0;

    auto header = [&](const LOp& o, std::vector<Instr>& pk) {
      uint32_t flags = o.has_out && o.opc != OP_OUT ? (uint32_t)F_OUT : 0u;
      uint32_t dst = NO_DST;
      if (o.val != 0xFFFFFFFFu && slot_of[o.val] >= 0) dst = (uint32_t)slot_of[o.val];
      auto slot = [&](uint32_t v) {
        if (slot_of[v] < 0) throw Error("latency plan: operand without a slot");
        return (uint32_t)slot_of[v];
      };
      auto inline_const = [&](const U256& v) {
        const uint32_t off = (uint32_t)pk.size();
        Instr lo4, hi4;
        lo4.x = v.l[0]; lo4.y = v.l[1]; lo4.z = v.l[2]; lo4.w = v.l[3];
        hi4.x = v.l[4]; hi4.y = v.l[5]; hi4.z = v.l[6]; hi4.w = v.l[7];
        pk.push_back(lo4); pk.push_back(hi4);
        return off;
      };
      if (o.opc == OP_INPUT) return make_instr(OP_INPUT, flags, dst, o.input, 0, o.out_pos);
      if (o.opc == OP_OUT) {
        if (o.in[0] < N && is_const[o.in[0]]) return make_instr(OP_OUT, F_A_CONST, NO_DST, inline_const(mp.const_val[o.in[0]]), 0, o.out_pos);
        return make_instr(OP_OUT, 0, NO_DST, slot(o.in[0]), 0, o.out_pos);
      }
      if (o.opc == OP_SHRAND) return make_instr(OP_SHRAND, flags, dst, slot(o.in[0]), o.shift | (inline_const(o.mask) << 8), o.out_pos);
      if (o.opc == OP_POW5) return make_instr(OP_POW5, flags, dst, slot(o.in[0]) | ((o.pos4 == NO_POS ? 0xFFFFu : o.pos4 - o.pos2) << 16), o.pos2, o.out_pos);
      if (o.opc == OP_POW4) return make_instr(OP_POW4, o.pos4 != NO_POS ? (uint32_t)F_OUT : 0u, dst, slot(o.in[0]), o.pos2, o.pos4 != NO_POS ? o.pos4 : 0u);
      if (o.opc == OP_DOT) {
        // terms ordered by kind so that the lanes of a warp walk the same code path
        std::vector<PTerm> ts = o.terms;
        std::stable_sort(ts.begin(), ts.end(), [](const PTerm& a, const PTerm& b) {
          auto key = [](const PTerm& t) { return t.kind == 0 ? 0 : t.kind == 1 ? (t.neg ? 2 : 1) : 3; };
          return key(a) < key(b);
        });
        const uint32_t tail = (uint32_t)pk.size();
        pk.resize(pk.size() + (ts.size() + 1) / 2, make_instr(OP_NOP, 0, 0, 0, 0, 0));
        std::vector<uint32_t> words;
        for (const PTerm& t : ts) {
          const uint32_t kind = t.kind == 0 ? (uint32_t)T_MAC : t.kind == 2 ? (uint32_t)T_CONST : (t.neg ? (uint32_t)T_SUBHI : (uint32_t)T_ADDHI);
          const uint32_t reg = t.kind == 2 ? 0u : slot(t.node);
          const uint32_t ci = t.kind == 1 ? 0u : inline_const(prescale(t.c, t.neg));
          words.push_back(kind | (reg << 16)); words.push_back(ci);
        }
        if (words.size() & 2) { words.push_back(0); words.push_back(0); }
        for (size_t k = 0; k < words.size(); k += 4) { Instr& sl = pk[tail + k / 4]; sl.x = words[k]; sl.y = words[k + 1]; sl.z = words[k + 2]; sl.w = words[k + 3]; }
        // shape hint for the kernel's straight-line path (.y bits 16..): 1-2 products, at most one added value, no
        // subtracted value, at most one constant -- the Poseidon mix layers; bit 0 = applies, bits 1-2 = number of
        // products, bit 3 = has an added value, bit 4 = has a constant.  Terms are already ordered MAC, +value, constant.
        uint32_t n_k[4] = {0, 0, 0, 0};
        for (const PTerm& t : ts) n_k[t.kind == 0 ? 0 : t.kind == 2 ? 3 : (t.neg ? 2 : 1)]++;
        uint32_t shape = 0;
        if (n_k[0] >= 1 && n_k[0] <= 2 && n_k[1] <= 1 && n_k[2] == 0 && n_k[3] <= 1) shape = 1u | (n_k[0] << 1) | (n_k[1] << 3) | (n_k[3] << 4);
        return make_instr(OP_DOT, flags, dst, (uint32_t)ts.size() | (o.ncs << 8) | (shape << 16), tail, o.out_pos);
      }
      uint32_t enc[3] = {0, 0, 0};
      for (int k = 0; k < o.n_in; k++) {
        if (o.in[k] < N && is_const[o.in[k]]) { enc[k] = inline_const(mp.const_val[o.in[k]]); flags |= (F_A_CONST << k); }
        else enc[k] = slot(o.in[k]);
      }
      return make_instr(o.opc, flags, dst, enc[0], enc[1], (o.opc == OP_TERN || o.opc == OP_MULADD) ? enc[2] : o.out_pos);
    };
    // header() emits offsets relative to the start of the instruction's own extras; a packet places them at `rb`
    auto rebase_header = [&](Instr h, uint32_t rb) {
      const uint32_t op = h.x & 0xFFu;
      if (op == OP_DOT) { h.z += rb; return h; }
      if (op == OP_SHRAND) { h.z = (h.z & 0xFFu) | (((h.z >> 8) + rb) << 8); return h; }
      if (op == OP_INPUT || op == OP_POW5 || op == OP_POW4) return h;
      if (h.x & F_A_CONST) h.y += rb;
      if ((h.x & F_B_CONST) && op_has_b_host(op)) h.z += rb;
      if ((h.x & F_C_CONST) && (op == OP_TERN || op == OP_MULADD)) h.w += rb;
      return h;
    };
    // appends a packet with the chains headed by list[from ..] to lp.code: at most 32 of them (one lane each), fewer
    // if the packet would exceed `cap` slots (0 = no limit).  Header k belongs to lane k mod lanes, so a lane finds the
    // instructions of its chain at k = lane, lane + lanes, ...; shorter chains are padded with OP_NOP.
    // returns {offset, slots, headers, lanes}
    // build_packet: the packet itself (pk_out), not yet placed; `reserve` = slots the caller appends behind it (they count
    // against `cap`).  returns {headers, chains taken}
    auto build_packet = [&](const std::vector<const LOp*>& list, size_t from, uint32_t cap, uint32_t reserve, std::vector<Instr>& pk) {
      size_t n = std::min<size_t>(32, list.size() - from);
      for (;; n = (n + 1) / 2) {
        size_t rows = n ? 1 : 0;
        for (size_t k = 0; k < n; k++) { size_t len = 0; for (const LOp* o = list[from + k]; o; o = o->chain_next >= 0 ? &ops[(size_t)o->chain_next] : nullptr) len++; rows = std::max(rows, len); }
        const uint32_t nh = (uint32_t)(rows * n);
        std::vector<Instr> hs(nh, make_instr(OP_NOP, 0, 0, 0, 0, 0)), extra, tmp;
        std::vector<uint32_t> ebase(nh, 0);
        for (size_t k = 0; k < n; k++) {
          size_t r = 0;
          for (const LOp* o = list[from + k]; o; o = o->chain_next >= 0 ? &ops[(size_t)o->chain_next] : nullptr, r++) {
            tmp.clear();
            hs[r * n + k] = header(*o, tmp);
            ebase[r * n + k] = (uint32_t)extra.size();
            extra.insert(extra.end(), tmp.begin(), tmp.end());
          }
        }
        pk.assign(1 + nh, make_instr(OP_NOP, 0, 0, 0, 0, 0));
        for (uint32_t i = 0; i < nh; i++) {
          const uint32_t rb = 1 + nh + ebase[i];       // where this header's extras start in the packet
          pk[1 + i] = rebase_header(hs[i], rb);
          if ((hs[i].x & 0xFFu) == OP_DOT) {            // the term slots of an OP_DOT tail carry constant offsets too
            const uint32_t nt = hs[i].y & 0xFFu;
            for (uint32_t t = 0; t < nt; t++) {
              Instr& sl = extra[ebase[i] + hs[i].z + (t >> 1)];
              uint32_t& lo_w = (t & 1) ? sl.z : sl.x; uint32_t& ci = (t & 1) ? sl.w : sl.y;
              const uint32_t kind = lo_w & 0xFu;
              if (kind == T_MAC || kind == T_CONST) ci += rb;
            }
          }
        }
        pk.insert(pk.end(), extra.begin(), extra.end());
        if (!cap || pk.size() + reserve <= cap || n <= 1) {
          if (cap && pk.size() + reserve > cap) throw Error("latency plan: one chain does not fit a packet");
          for (uint32_t i = 0; i < nh; i++) lp.n_instrs += (hs[i].x & 0xFFu) != OP_NOP;
          return std::array<uint32_t, 2>{nh, (uint32_t)n};
        }
      }
    };
    auto emit_packet = [&](const std::vector<const LOp*>& list, size_t from, uint32_t cap) {
      size_t n = std::min<size_t>(32, list.size() - from);
      std::vector<Instr> pk;
      for (;; n = (n + 1) / 2) {
        size_t rows = n ? 1 : 0;
        for (size_t k = 0; k < n; k++) { size_t len = 0; for (const LOp* o = list[from + k]; o; o = o->chain_next >= 0 ? &ops[(size_t)o->chain_next] : nullptr) len++; rows = std::max(rows, len); }
        const uint32_t nh = (uint32_t)(rows * n);
        std::vector<Instr> hs(nh, make_instr(OP_NOP, 0, 0, 0, 0, 0)), extra, tmp;
        std::vector<uint32_t> ebase(nh, 0);
        for (size_t k = 0; k < n; k++) {
          size_t r = 0;
          for (const LOp* o = list[from + k]; o; o = o->chain_next >= 0 ? &ops[(size_t)o->chain_next] : nullptr, r++) {
            tmp.clear();
            hs[r * n + k] = header(*o, tmp);
            ebase[r * n + k] = (uint32_t)extra.size();
            extra.insert(extra.end(), tmp.begin(), tmp.end());
          }
        }
        pk.assign(1 + nh, make_instr(OP_NOP, 0, 0, 0, 0, 0));
        for (uint32_t i = 0; i < nh; i++) {
          const uint32_t rb = 1 + nh + ebase[i];       // where this header's extras start in the packet
          pk[1 + i] = rebase_header(hs[i], rb);
          if ((hs[i].x & 0xFFu) == OP_DOT) {            // the term slots of an OP_DOT tail carry constant offsets too
            const uint32_t nt = hs[i].y & 0xFFu;
            for (uint32_t t = 0; t < nt; t++) {
              Instr& sl = extra[ebase[i] + hs[i].z + (t >> 1)];
              uint32_t& lo_w = (t & 1) ? sl.z : sl.x; uint32_t& ci = (t & 1) ? sl.w : sl.y;
              const uint32_t kind = lo_w & 0xFu;
              if (kind == T_MAC || kind == T_CONST) ci += rb;
            }
          }
        }
        pk.insert(pk.end(), extra.begin(), extra.end());
        if (!cap || pk.size() <= cap || n <= 1) {
          if (cap && pk.size() > cap) throw Error("latency plan: one chain does not fit a packet");
          const uint32_t off = (uint32_t)lp.code.size();
          lp.code.insert(lp.code.end(), pk.begin(), pk.end());
          for (uint32_t i = 0; i < nh; i++) lp.n_instrs += (hs[i].x & 0xFFu) != OP_NOP;
          return std::array<uint32_t, 5>{off, (uint32_t)pk.size(), nh, (uint32_t)n, (uint32_t)n};
        }
      }
    };

    if (lo.dataflow) {
      // ---- 3'. dataflow plan: per-warp instruction streams, no level barrier --------------------------------------
      // Every warp (main and slow alike) walks its own stream of packets in order; a packet names, per other warp, how
      // many of that warp's packets must be complete before it may start (operands produced there, and readers there
      // of the values whose slots it overwrites).  Levels survive only as the order of emission, which is what makes
      // the waits acyclic: a packet only ever waits for packets emitted before it, and a warp runs its packets in the
      // order of emission.  A simple timing model (finish time per packet) steers the warp assignment.
      // Physical warps: a warp's SM sub-partition (its own multiplier pipe) is its index mod 4.  Warp 0 takes the most
      // critical instructions of every level and keeps its sub-partition to itself: warps 4 and 8 stay empty (measured:
      // three warps of dependent carry chains on one sub-partition run 1.5x slower each, profiles/r02n).
      std::vector<uint32_t> phys;                          // logical warp (mains first, then slows) -> physical warp
      for (uint32_t skip = lo.exclusive_warp0 ? 2u : 0u;; skip--) {       // leave warps 4 and 8 empty, or only 4, or none: whatever fits 12 warps
        phys.clear();
        for (uint32_t id = 0; phys.size() < lo.n_warps + lo.n_slow_warps; id++) if (!(id > 0 && id % 4 == 0 && id / 4 <= skip)) phys.push_back(id);
        if (phys.back() < 12 || skip == 0) break;
      }
      const uint32_t NW = phys.back() + 1;
      if (NW > 12) throw Error("latency plan: more than 12 warps");
      const uint32_t C = lo.packet_slots, WV = 3;          // chunk capacity (16 B slots); slots of a wait vector (12 words)
      // cycles, measured in place per packet with 6 + 3 warps on the SM (profiles/r02p/clocks_authv2.summary.txt: medians
      // from after the wait to the publish, interpreter included): about 650 cycles of fetch / decode / stores around the
      // arithmetic, and the arithmetic itself 1.3 - 1.5x slower than alone on the SM
      const uint64_t HOP = 150, ROW = 300;                 // a value crossing warps (publish + poll); descriptor + wait between two packets
      auto df_cost = [&](const LOp& o) -> uint64_t {
        switch (o.opc) {
          case OP_MUL: return 1870; case OP_SQR: return 1580; case OP_POW5: return 3420; case OP_POW4: return 2510; case OP_MULADD: return 1950;
          case OP_DOT: { uint32_t n = 0; for (const PTerm& t : o.terms) n += t.kind == 0; return 1300 + 750ull * n + 60ull * (uint32_t)o.terms.size(); }
          case OP_ADD: case OP_SUB: return 720;
          case OP_DIV: return 53700; case OP_INV: return 52700; case OP_POW: return 500000; case OP_IDIV: case OP_MOD: return 50000;
          default: return 700;
        }
      };
      const size_t NO = ops.size();
      std::vector<int32_t> def_of(NV, -1);
      for (size_t k = 0; k < NO; k++) if (ops[k].val != 0xFFFFFFFFu) def_of[ops[k].val] = (int32_t)k;
      std::vector<uint64_t> blevel(NO, 0);                 // longest path from the start of the instruction to a sink
      for (size_t k = 0; k < NO; k++) blevel[k] = df_cost(ops[k]);
      for (size_t k = NO; k-- > 0;)
        for_operands(ops[k], [&](uint32_t v) { const int32_t d = def_of[v]; if (d >= 0) blevel[(size_t)d] = std::max(blevel[(size_t)d], df_cost(ops[(size_t)d]) + blevel[k]); });
      std::vector<std::vector<Instr>> stream(NW);
      std::vector<uint32_t> fill(NW, 0);                   // slots used in the current chunk of each stream
      std::vector<uint32_t> n_rows(NW, 0);
      std::vector<std::vector<uint64_t>> row_finish(NW);   // timing model: finish time of packet r (0-based) of warp w
      std::vector<uint64_t> t_warp(NW, 0);
      std::vector<std::array<uint32_t, 12>> known(NW);     // what each warp has already waited for
      for (auto& k : known) k.fill(0);
      std::vector<uint32_t> prod_w(NV, 0xFFFFFFFFu), prod_r(NV, 0);   // producer (warp, 1-based packet number) of each value
      std::vector<std::array<uint32_t, 12>> slot_busy;     // per slot: per warp, the last packet that touches its current value
      std::vector<std::array<uint32_t, 12>> war_of(NO);    // per instruction: the busy vector of its destination slot's previous value
      std::vector<uint32_t> fifo;                          // free slots, oldest first: their readers finished long ago
      size_t fifo_head = 0;
      const std::array<uint32_t, 12> zero12 = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
      auto ready_time = [&](const LOp& o, uint32_t w) {
        uint64_t t = 0;
        for_operands(o, [&](uint32_t v) { if (prod_w[v] != 0xFFFFFFFFu) t = std::max(t, row_finish[prod_w[v]][prod_r[v] - 1] + (prod_w[v] != w ? HOP : 0)); });
        return t;
      };
      auto close_chunk = [&](uint32_t w) {
        if (fill[w] == 0) return;
        // terminator descriptor (size 0) if there is room, then padding up to the chunk boundary
        while (fill[w] < C) { stream[w].push_back(make_instr(OP_NOP, 0, 0, 0, 0, 0)); stream[w].back().x = 0; fill[w]++; }
        fill[w] = 0;
      };
      // emits the instructions list[from ..] (one class, independent) as packets of warp w; returns how many it took
      auto emit_df = [&](uint32_t w, const std::vector<const LOp*>& list, size_t from, uint64_t cost) {
        // requirement vector: producers of the operands, and whoever touched the previous values of the destination slots
        std::array<uint32_t, 12> req = zero12;
        std::vector<Instr> pk;
        const auto bp = build_packet(list, from, C, WV, pk);
        const size_t n = bp[1];
        for (size_t k = 0; k < n; k++) {
          const LOp& o = *list[from + k];
          for_operands(o, [&](uint32_t v) { if (prod_w[v] != 0xFFFFFFFFu && prod_w[v] != w) req[prod_w[v]] = std::max(req[prod_w[v]], prod_r[v]); });
          const std::array<uint32_t, 12>& wr = war_of[(size_t)(&o - ops.data())];
          for (uint32_t x = 0; x < NW; x++) if (x != w) req[x] = std::max(req[x], wr[x]);
        }
        bool need = false;
        for (uint32_t x = 0; x < NW; x++) { if (req[x] > known[w][x]) { need = true; known[w][x] = req[x]; } }
        uint32_t wait_off = 0;
        if (need) {
          wait_off = (uint32_t)pk.size();
          for (uint32_t q = 0; q < WV; q++) { Instr sl; sl.x = known[w][4 * q]; sl.y = known[w][4 * q + 1]; sl.z = known[w][4 * q + 2]; sl.w = known[w][4 * q + 3]; pk.push_back(sl); }
        }
        if (pk.size() > C) throw Error("latency plan: packet larger than a chunk");
        if (fill[w] + pk.size() > C) close_chunk(w);
        const uint32_t row = ++n_rows[w];
        pk[0].x = (uint32_t)pk.size(); pk[0].y = bp[0] | ((uint32_t)n << 16); pk[0].z = wait_off; pk[0].w = row;
        stream[w].insert(stream[w].end(), pk.begin(), pk.end());
        fill[w] += (uint32_t)pk.size();
        if (fill[w] == C) fill[w] = 0;
        // timing model
        uint64_t start = t_warp[w];
        if (need) for (uint32_t x = 0; x < NW; x++) if (x != w && req[x]) start = std::max(start, row_finish[x][req[x] - 1] + HOP);
        for (size_t k = 0; k < n; k++) start = std::max(start, ready_time(*list[from + k], w));
        const uint64_t end = start + ROW + cost;
        t_warp[w] = end; row_finish[w].push_back(end);
        // bookkeeping: producers, slot users
        for (size_t k = 0; k < n; k++) {
          const LOp& o = *list[from + k];
          for_operands(o, [&](uint32_t v) { if (slot_of[v] >= 0) slot_busy[(size_t)slot_of[v]][w] = std::max(slot_busy[(size_t)slot_of[v]][w], row); });
          if (o.val != 0xFFFFFFFFu) { prod_w[o.val] = w; prod_r[o.val] = row; if (slot_of[o.val] >= 0) slot_busy[(size_t)slot_of[o.val]][w] = std::max(slot_busy[(size_t)slot_of[o.val]][w], row); }
        }
        lp.n_rows++;
        lp.n_waits_df += need;
        return n;
      };
      std::vector<uint32_t> mains, slows;
      for (uint32_t L = 0; L < n_levels; L++) {
        mains.clear(); slows.clear();
        for (uint32_t k : by_level[L]) { if (ops[k].slow) slows.push_back(k); else mains.push_back(k); }
        // destination slots of everything issued at this level; the previous value's users become the instruction's WAR waits
        for (uint32_t k : by_level[L]) {
          const LOp& o = ops[k];
          war_of[k] = zero12;
          if (o.val == 0xFFFFFFFFu || last_use[o.val] < 0) continue;
          uint32_t sl;
          if (fifo_head < fifo.size()) { sl = fifo[fifo_head++]; war_of[k] = slot_busy[sl]; slot_busy[sl] = zero12; }
          else { sl = n_slots++; slot_busy.push_back(zero12); if (n_slots > lo.max_slots) throw Error("latency plan: graph is too wide for the shared-memory value file"); }
          slot_of[o.val] = (int32_t)sl;
          dying[(size_t)last_use[o.val]].push_back(o.val);
        }
        // bundles: one class, operands ready at about the same time, at most 32; the most critical bundle picks its warp first
        struct It { uint64_t cls, cost, ready, bl; const LOp* op; };
        std::vector<It> items;
        for (uint32_t k : mains) items.push_back({lat_class(ops[k]), df_cost(ops[k]), ready_time(ops[k], 0xFFFFFFFFu), blevel[k], &ops[k]});
        std::stable_sort(items.begin(), items.end(), [](const It& a, const It& b) { return a.cls != b.cls ? a.cls < b.cls : a.ready < b.ready; });
        struct Bundle { size_t a, b; uint64_t bl; };
        std::vector<Bundle> bundles;
        for (size_t a = 0; a < items.size();) {
          size_t b = a; uint64_t bl = 0;
          while (b < items.size() && b - a < 32 && items[b].cls == items[a].cls && items[b].ready <= items[a].ready + 400) { bl = std::max(bl, items[b].bl); b++; }
          bundles.push_back({a, b, bl});
          a = b;
        }
        std::stable_sort(bundles.begin(), bundles.end(), [](const Bundle& x, const Bundle& y) { return x.bl > y.bl; });
        const uint64_t level_bl = bundles.empty() ? 0 : bundles[0].bl;
        std::vector<const LOp*> list;
        uint32_t width = 0;
        for (const Bundle& bd : bundles) {
          list.clear();
          for (size_t k = bd.a; k < bd.b; k++) list.push_back(items[k].op);
          width += (uint32_t)list.size();
          // warp 0 is reserved for the critical bundles of the level (those on the longest remaining path)
          const bool critical = !lo.exclusive_warp0 || lo.n_warps == 1 || bd.bl * 100 >= level_bl * 98;
          uint32_t best = phys[critical ? 0 : 1]; uint64_t best_end = ~0ull;
          for (uint32_t lw = critical ? 0 : 1; lw < lo.n_warps; lw++) {
            const uint32_t w = phys[lw];
            uint64_t rdy = 0;
            for (const LOp* o : list) rdy = std::max(rdy, ready_time(*o, w));
            const uint64_t end = std::max(t_warp[w], rdy) + ROW + items[bd.a].cost;
            if (end < best_end) { best_end = end; best = w; }
          }
          for (size_t from = 0; from < list.size();) from += emit_df(best, list, from, items[bd.a].cost);
        }
        lp.max_level_width = std::max(lp.max_level_width, width);
        // long ops: packets of up to 32 lanes of one opcode on the slow warp that is free first
        std::stable_sort(slows.begin(), slows.end(), [&](uint32_t a, uint32_t b) { return ops[a].opc < ops[b].opc; });
        for (size_t a = 0; a < slows.size();) {
          size_t b = a;
          while (b < slows.size() && b - a < 32 && ops[slows[b]].opc == ops[slows[a]].opc) b++;
          list.clear();
          for (size_t k = a; k < b; k++) list.push_back(&ops[slows[k]]);
          uint32_t best = phys[lo.n_warps]; uint64_t best_end = ~0ull;
          for (uint32_t lw = lo.n_warps; lw < lo.n_warps + lo.n_slow_warps; lw++) {
            const uint32_t w = phys[lw];
            uint64_t rdy = 0;
            for (const LOp* o : list) rdy = std::max(rdy, ready_time(*o, w));
            const uint64_t end = std::max(t_warp[w], rdy);
            if (end < best_end) { best_end = end; best = w; }
          }
          for (size_t from = 0; from < list.size();) from += emit_df(best, list, from, df_cost(*list[0]));
          a = b;
        }
        for (uint32_t v : dying[L]) fifo.push_back((uint32_t)slot_of[v]);
      }
      // streams -> code: whole chunks, back to back
      lp.dataflow = true; lp.chunk_slots = C;
      lp.stream_off.assign(NW, 0); lp.stream_chunks.assign(NW, 0);
      for (uint32_t w = 0; w < NW; w++) {
        close_chunk(w);
        lp.stream_off[w] = (uint32_t)lp.code.size();
        lp.stream_chunks[w] = (uint32_t)(stream[w].size() / C);
        lp.code.insert(lp.code.end(), stream[w].begin(), stream[w].end());
      }
      for (uint32_t w = 0; w < NW; w++) lp.est_cycles = std::max<uint64_t>(lp.est_cycles, t_warp[w]);
      lp.n_levels = n_levels;
      lp.n_slots = std::max(n_slots, 1u);
      lp.n_phys_warps = NW;
      return lp;
    }
    std::vector<uint32_t> mains, slows;
    for (uint32_t L = 0; L < n_levels; L++) {
      mains.clear(); slows.clear();
      for (uint32_t k : by_level[L]) { if (ops[k].slow) slows.push_back(k); else if (ops[k].chain_prev < 0) mains.push_back(k); }
      // destination slots of everything issued at this level
      for (uint32_t k : by_level[L]) {
        const LOp& o = ops[k];
        if (o.val == 0xFFFFFFFFu || last_use[o.val] < 0) continue;
        uint32_t s;
        if (!free_slots.empty()) { s = free_slots.back(); free_slots.pop_back(); }
        else { s = n_slots++; if (n_slots > lo.max_slots) throw Error("latency plan: graph is too wide for the shared-memory value file"); }
        slot_of[o.val] = (int32_t)s;
        dying[(size_t)last_use[o.val]].push_back(o.val);
      }
      // long ops: jobs of up to 32 lanes of one opcode, queued to the least busy slow warp
      std::stable_sort(slows.begin(), slows.end(), [&](uint32_t a, uint32_t b) { return ops[a].opc < ops[b].opc; });
      for (size_t a = 0; a < slows.size();) {
        size_t b = a;
        while (b < slows.size() && b - a < 32 && ops[slows[b]].opc == ops[slows[a]].opc) b++;
        // least busy slow warp; ties go to the highest index: the heaviest instruction classes of a level sit on main
        // warps 0, 1, .. and a warp's SM sub-partition is its index mod 4, so the long jobs keep away from them
        uint32_t w = lo.n_slow_warps - 1;
        for (uint32_t x = lo.n_slow_warps - 1; x-- > 0;) if (busy[x] < busy[w]) w = x;
        busy[w] = std::max<uint64_t>(busy[w], L) + D;
        std::vector<const LOp*> jl;
        for (size_t k = a; k < b; k++) jl.push_back(&ops[slows[k]]);
        const auto jp = emit_packet(jl, 0, 0);
        if (jp[3] != b - a) throw Error("latency plan: slow job packet");
        jobq[w].push_back({n_phys, jp[0], (uint32_t)(b - a)});
        const uint32_t wl = L + D - 1;
        if (wl >= n_levels) throw Error("latency plan: wait level out of range");
        pending_waits[wl].push_back({w, (uint32_t)jobq[w].size()});
        a = b;
      }
      // bundles: <= 32 instructions of one class; longest bundle first onto the least loaded warp.  Two warps on the
      // same SM sub-partition (warp index mod 4) share one multiplier pipe, which is counted as partial contention.
      struct Item { uint64_t cls; uint32_t cost; const LOp* op; };
      std::vector<Item> items;
      for (uint32_t k : mains) {
        uint64_t cls = 0; uint32_t cost = 0;
        for (const LOp* o = &ops[k]; o; o = o->chain_next >= 0 ? &ops[(size_t)o->chain_next] : nullptr) { cls = cls * 0x9E3779B97F4A7C15ull + lat_class(*o) + 1; cost += lat_cost(*o); }
        items.push_back({cls, cost, &ops[k]});
      }
      std::stable_sort(items.begin(), items.end(), [](const Item& a, const Item& b) { return a.cost != b.cost ? a.cost > b.cost : a.cls < b.cls; });
      std::vector<std::vector<const LOp*>> per_warp(lo.n_warps);
      std::vector<double> load(lo.n_warps, 0.0);
      for (size_t a = 0; a < items.size();) {
        size_t b = a;
        while (b < items.size() && b - a < 32 && items[b].cls == items[a].cls) b++;
        uint32_t best = 0; double best_t = 1e300;
        for (uint32_t w = 0; w < lo.n_warps; w++) {
          double t = load[w] + items[a].cost;
          for (uint32_t x = w & 3u; x < lo.n_warps; x += 4) if (x != w) t += 0.4 * std::min<double>(load[x], items[a].cost);
          if (t < best_t) { best_t = t; best = w; }
        }
        load[best] += items[a].cost;
        for (size_t k = a; k < b; k++) per_warp[best].push_back(items[k].op);
        a = b;
      }
      double worst = 0;
      uint32_t width = 0;
      for (uint32_t w = 0; w < lo.n_warps; w++) { worst = std::max(worst, load[w]); width += (uint32_t)per_warp[w].size(); }
      // physical levels: every packet must fit one stage of the kernel's shared-memory ring, so a wide level is cut
      // into several consecutive ones (all its operands are older, all its destinations are fresh: no hazard)
      {
        std::vector<size_t> done(lo.n_warps, 0);
        bool more = true;
        while (more) {
          more = false;
          for (uint32_t w = 0; w < lo.n_warps; w++) {
            const auto pp = emit_packet(per_warp[w], done[w], lo.packet_slots);
            done[w] += pp[4];
            pinfo.push_back({pp[0], pp[1], pp[2], pp[3]});
            more |= done[w] < per_warp[w].size();
          }
          n_phys++;
        }
      }
      for (const auto& pw : pending_waits[L]) { lp.waits.push_back(n_phys - 1); lp.waits.push_back(pw[0]); lp.waits.push_back(pw[1]); lp.waits.push_back(0); }
      lp.est_cycles += (uint64_t)worst + LAT_LEVEL_OVERHEAD;
      if (dbg_level >= 0 && L >= (uint32_t)dbg_level && L < (uint32_t)dbg_level + dbg_count) {      // GW_LAT_DEBUG=<level>: dump 24 (GW_LAT_DEBUG_N) levels of the schedule
        fprintf(stderr, "L%u worst %.0f:", L, worst);
        for (uint32_t w = 0; w < lo.n_warps; w++) { fprintf(stderr, " w%u[", w); for (const LOp* o : per_warp[w]) fprintf(stderr, "%llx ", (unsigned long long)lat_class(*o)); fprintf(stderr, "]"); }
        fprintf(stderr, "\n");
      }
      lp.max_level_width = std::max(lp.max_level_width, width);
      // slots read for the last time in this level become reusable from the next level on
      for (uint32_t v : dying[L]) free_slots.push_back((uint32_t)slot_of[v]);
    }

    // ---- 4. descriptors: the packet of (L, w) names the packet of (L + 2, w); the first two come from `first` ----
    for (uint32_t L = 0; L < n_phys; L++)
      for (uint32_t w = 0; w < lo.n_warps; w++) {
        Instr& d = lp.code[pinfo[(size_t)L * lo.n_warps + w][0]];
        if (L + 2 < n_phys) { const auto& nx = pinfo[(size_t)(L + 2) * lo.n_warps + w]; d.x = nx[0]; d.y = nx[1]; d.z = nx[2]; d.w = nx[3]; }
        else { d.x = d.y = d.z = d.w = 0; }
      }
    lp.first.assign((size_t)lo.n_warps * 8, 0);
    for (uint32_t w = 0; w < lo.n_warps; w++)
      for (uint32_t j = 0; j < 2 && j < n_phys; j++)
        for (int k = 0; k < 4; k++) lp.first[(size_t)w * 8 + j * 4 + k] = pinfo[(size_t)j * lo.n_warps + w][k];
    lp.max_jobs = 1;
    for (const auto& q : jobq) lp.max_jobs = std::max<uint32_t>(lp.max_jobs, (uint32_t)q.size());
    lp.jobs.assign((size_t)lo.n_slow_warps * lp.max_jobs * 4, 0);
    lp.n_jobs.assign(lo.n_slow_warps, 0);
    for (uint32_t w = 0; w < lo.n_slow_warps; w++) {
      lp.n_jobs[w] = (uint32_t)jobq[w].size();
      for (size_t j = 0; j < jobq[w].size(); j++) {
        uint32_t* e = &lp.jobs[((size_t)w * lp.max_jobs + j) * 4];
        e[0] = jobq[w][j][0]; e[1] = jobq[w][j][1]; e[2] = jobq[w][j][2]; e[3] = 0;
      }
    }
    lp.n_levels = n_phys;
    lp.n_slots = std::max(n_slots, 1u);
    return lp;
  };

  // D from the cost model: one inversion spans about (its cycles / an average level) levels
  auto plan_for = [&](bool chain) {
    use_chain = chain;
    if (lo.slow_levels) return schedule(lo.slow_levels);
    LatencyPlan first = schedule(24);
    if (first.n_slow == 0) return first;
    const double avg = std::max(200.0, (double)first.est_cycles / std::max(1u, first.n_levels));
    // (dataflow plan: nothing waits at level boundaries, but a reader placed early in its warp's stream blocks what
    // follows it until the long operation is done -- twice the distance measured best on authV2, profiles/r02q)
    const uint32_t D = (uint32_t)std::min(4096.0, std::max(2.0, (lo.dataflow ? 2.0 * 53700.0 : 42000.0) / avg + 2.0));
    return schedule(D);
  };
  // chains trade levels for lane parallelism (instructions of different shapes cannot share a warp): keep whichever
  // schedule the cost model likes better (Poseidon / EdDSA graphs: chains; bit-level graphs like SHA-256: none)
  LatencyPlan a = plan_for(false);
  a.n_sbox_links = n_links;
  if (!lo.chain || lo.dataflow) return a;      // dataflow: an S-box is one OP_POW5 already; other chains would only serialise a lane
  LatencyPlan b = plan_for(true);
  b.n_sbox_links = n_links;
  return b.est_cycles < a.est_cycles ? b : a;
}

}  // namespace gw
