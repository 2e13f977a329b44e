// TEST-ONLY host simulator of the device plan: executes the instruction stream that plan.cpp emits
// with the host path of csrc/alu.cuh, one witness at a time.  It exists so that the graph codec, the
// inputs parser, the register allocator / spill logic and the op semantics can be checked against the
// oracle on a machine without a GPU.  It is NOT part of libcircom_witnesscalc.so (the product has no
// CPU fallback); the same alu_exec() runs on the device inside eval_batch_kernel.
#include <string.h>

#include <map>
#include <memory>

#include "../../circom-witnesscalc_b200/csrc/alu.cuh"
#include "../../circom-witnesscalc_b200/csrc/graph.hpp"
#include "../../circom-witnesscalc_b200/csrc/inputs.hpp"
#include "../../circom-witnesscalc_b200/csrc/plan.hpp"
#include "../../circom-witnesscalc_b200/csrc/wtns.hpp"

using namespace gw;

static bool lat_is_slow_op(uint32_t op) { return op == OP_DIV || op == OP_INV || op == OP_POW || op == OP_IDIV || op == OP_MOD; }
static bool op_has_b_host(uint32_t op) { return op < 32 || op == OP_TERN || op == OP_MULADD; }

struct SimGraph {
  Graph g; Plan plan; std::string err;
  // the latency plan of the last sim_eval_latency3 call and the options it was compiled under (one compilation per option set)
  std::vector<uint32_t> lat_key; LatencyPlan lat; bool lat_ok = false;
};

static fe to_fe(const U256& v) { fe r; memcpy(r.l, v.l, 32); return r; }

extern "C" {

// flags: bit 0 = fuse linear combinations (OP_DOT), bit 1 = narrow typing OFF, bit 2 = OP_POW5 fusion OFF,
// bits 8..15 = div_batch, bits 16..23 = max_terms (0 -> default, like GW_DIV_BATCH / GW_MAX_TERMS unset)
SimGraph* sim_load2(const uint8_t* data, size_t len, uint32_t n_regs, int flags, char* err, size_t errlen);
SimGraph* sim_load(const uint8_t* data, size_t len, uint32_t n_regs, char* err, size_t errlen) {
  return sim_load2(data, len, n_regs, 1, err, errlen);
}
SimGraph* sim_load2(const uint8_t* data, size_t len, uint32_t n_regs, int flags, char* err, size_t errlen) {
  try {
    std::unique_ptr<SimGraph> s(new SimGraph());
    s->g = deserialize_witnesscalc_graph(data, len);
    PlanOptions o; o.n_regs = n_regs; o.fuse_dot = (flags & 1) != 0; o.narrow = (flags & 2) == 0; o.fuse_pow5 = (flags & 4) == 0;
    if ((flags >> 8) & 0xFF) o.div_batch = (uint32_t)((flags >> 8) & 0xFF);
    if ((flags >> 16) & 0xFF) o.max_terms = (uint32_t)((flags >> 16) & 0xFF);
    s->plan = compile_plan(s->g, o);
    return s.release();
  } catch (const std::exception& e) { if (err && errlen) { strncpy(err, e.what(), errlen - 1); err[errlen - 1] = 0; } return nullptr; }
}
void sim_free(SimGraph* s) { delete s; }
// the compiled program: copies up to cap slots (4 words each: x, y, z, w) and returns the number of slots
size_t sim_code(SimGraph* s, uint32_t* out, size_t cap) {
  const std::vector<Instr>& c = s->plan.code;
  for (size_t i = 0; i < c.size() && i < cap; i++) { out[4 * i] = c[i].x; out[4 * i + 1] = c[i].y; out[4 * i + 2] = c[i].z; out[4 * i + 3] = c[i].w; }
  return c.size();
}
void sim_info2(SimGraph* s, uint64_t* out) { out[0] = s->plan.stats.narrow_instrs; out[1] = s->plan.stats.op_count[OP_WIDEN]; out[2] = s->plan.n_spill_narrow; out[3] = s->plan.stats.pow5; }
void sim_info(SimGraph* s, uint64_t* out) {
  const PlanStats& st = s->plan.stats;
  out[0] = s->g.nodes.size(); out[1] = s->plan.n_inputs; out[2] = s->plan.n_witness; out[3] = st.instrs;
  out[4] = s->plan.n_regs; out[5] = s->plan.n_spill; out[6] = st.spill_ld; out[7] = st.spill_st;
  out[8] = st.max_live; out[9] = s->plan.consts.size(); out[10] = st.live_ops; out[11] = st.graph_ops;
  out[12] = st.op_count[OP_DOT]; out[13] = st.dot_terms[T_MAC]; out[14] = st.inversions; out[15] = st.div_nodes;
  out[16] = st.slots; out[17] = st.op_count[OP_MUL] + st.op_count[OP_SQR]; out[18] = st.op_count[OP_ADD] + st.op_count[OP_SUB];
}
// inputs: I x 32 B, witness: W x 32 B; returns status bits, or -1 on a malformed plan
int64_t sim_eval(SimGraph* s, const uint8_t* inputs, uint8_t* witness) {
  const Plan& p = s->plan;
  std::vector<fe> rf(p.n_regs, fe_zero()), spill(p.n_spill, fe_zero());
  std::vector<int64_t> nspill(p.n_spill_narrow, 0);
  uint32_t st = 0;
  // value of one instruction from the CURRENT register file (no writes); false on a malformed instruction
  auto compute = [&](const Instr& ins, const Instr* tail, fe* out) {
    const uint32_t op = ins.x & 0xFF;
    fe A = fe_zero(), B = fe_zero(), C = fe_zero();
    auto load = [&](uint32_t idx, bool is_const, fe* o) { if (is_const) { if (idx >= p.consts.size()) return false; *o = to_fe(p.consts[idx]); } else { if (idx >= p.n_regs) return false; *o = rf[idx]; } return true; };
    if (op == OP_SPILL_LD) { if (ins.y >= p.n_spill) return false; *out = spill[ins.y]; return true; }
    if (op == OP_INPUT) {
      if (ins.y >= p.n_inputs) return false;
      fe v; memcpy(v.l, inputs + 32 * (size_t)ins.y, 32);
      *out = fe_reduce256(v); return true;
    }
    if (op == OP_DOT) {
      const uint32_t nt = ins.y & 0xFF, ncs = (ins.y >> 8) & 0xFF;
      if (nt == 0 || nt > DOT_MAX_TERMS || ncs < 1 || ncs > 3) return false;
      dot_acc P; dot_init(P);
      for (uint32_t t = 0; t < nt; t++) {
        const Instr& sl = tail[t >> 1];
        const uint32_t lo = (t & 1) ? sl.z : sl.x, ci = (t & 1) ? sl.w : sl.y;
        const uint32_t kind = lo & 0xF, reg = lo >> 16;
        if (kind > T_CONST || reg >= p.n_regs || ci >= p.consts.size()) return false;
        dot_term(P, kind, rf[reg], to_fe(p.consts[ci]));
      }
      *out = fe_mont_reduce(P, (int)ncs); return true;
    }
    if (op == OP_SHRAND) {
      if (ins.y >= p.n_regs || (ins.z >> 8) >= p.consts.size()) return false;
      *out = fe_shr_and(rf[ins.y], ins.z & 0xFF, to_fe(p.consts[ins.z >> 8])); return true;
    }
    if (!load(ins.y, ins.x & F_A_CONST, &A)) return false;
    if (op == OP_OUT) { *out = A; return true; }
    if (op_has_b(op) && !load(ins.z, ins.x & F_B_CONST, &B)) return false;
    if (op == OP_TERN && !load(ins.w, ins.x & F_C_CONST, &C)) return false;
    *out = alu_exec(op, A, B, C, st);
    return true;
  };
  auto commit = [&](const Instr& ins, const fe& R) {
    const uint32_t op = ins.x & 0xFF, dst = ins.x >> 16;
    if (op == OP_OUT) { if (ins.w >= p.n_witness) return false; memcpy(witness + 32 * (size_t)ins.w, R.l, 32); return true; }
    if (dst != NO_DST) { if (dst >= p.n_regs) return false; rf[dst] = R; }
    if (ins.x & F_OUT) { if (ins.w >= p.n_witness) return false; memcpy(witness + 32 * (size_t)ins.w, R.l, 32); }
    return true;
  };
  // narrow instructions (isa.h: F_NARROW): int64 in limbs 0..1; limbs 2..7 of a narrow register are poisoned here
  // so that any wide read of a narrow value (a plan compiler bug) shows up as a wrong witness
  auto nload = [&](uint32_t idx, bool is_const, int64_t* o) {
    if (is_const) { if (idx >= p.consts.size()) return false; *o = narrow_of(to_fe(p.consts[idx])); }
    else { if (idx >= p.n_regs) return false; *o = narrow_of(rf[idx]); }
    return true;
  };
  auto poison = [&](int64_t v) { fe r; r.l[0] = (uint32_t)(uint64_t)v; r.l[1] = (uint32_t)((uint64_t)v >> 32); for (int i = 2; i < 8; i++) r.l[i] = 0xDEADBEEFu; return r; };
  auto narrow_step = [&](const Instr& ins, const Instr* tail) {
    const uint32_t op = ins.x & 0xFF, dst = ins.x >> 16;
    int64_t r = 0, a = 0, b = 0, c = 0;
    if (op == OP_SPILL_ST) { if (ins.y >= p.n_regs || ins.z >= p.n_spill_narrow) return false; nspill[ins.z] = narrow_of(rf[ins.y]); return true; }
    if (op == OP_OUT) {
      if (!nload(ins.y, false, &a) || ins.w >= p.n_witness) return false;
      fe v = fe_from_narrow(a); memcpy(witness + 32 * (size_t)ins.w, v.l, 32); return true;
    }
    if (op == OP_SPILL_LD) { if (ins.y >= p.n_spill_narrow) return false; r = nspill[ins.y]; }
    else if (op == OP_DOT) {
      const uint32_t nt = ins.y & 0xFF;
      if (nt == 0 || nt > DOT_MAX_TERMS) return false;
      for (uint32_t t = 0; t < nt; t++) {
        const Instr& sl = tail[t >> 1];
        const uint32_t lo = (t & 1) ? sl.z : sl.x, ci = (t & 1) ? sl.w : sl.y;
        const uint32_t kind = lo & 0xF, reg = lo >> 16;
        int64_t x = 0, cc = 0;
        if (kind > T_CONST) return false;
        if (kind != T_CONST && !nload(reg, false, &x)) return false;
        if ((kind == T_MAC || kind == T_CONST) && !nload(ci, true, &cc)) return false;
        r = narrow_dot_term(r, kind, x, cc);
      }
    } else if (op == OP_SHRAND) {
      if (!nload(ins.y, false, &a) || !nload(ins.z >> 8, true, &c)) return false;
      r = narrow_shr_and(a, ins.z & 0xFF, c);
    } else {
      if (!nload(ins.y, ins.x & F_A_CONST, &a)) return false;
      if (op_has_b(op) && !nload(ins.z, ins.x & F_B_CONST, &b)) return false;
      if (op == OP_TERN && !nload(ins.w, ins.x & F_C_CONST, &c)) return false;
      r = narrow_exec(op, a, b, c);
    }
    if (dst != NO_DST) { if (dst >= p.n_regs) return false; rf[dst] = poison(r); }
    if (ins.x & F_OUT) { if (ins.w >= p.n_witness) return false; fe v = fe_from_narrow(r); memcpy(witness + 32 * (size_t)ins.w, v.l, 32); }
    return true;
  };
  for (size_t pc = 0; pc < p.code.size();) {
    const Instr& ins = p.code[pc];
    const uint32_t len = instr_slots(ins);
    if (pc + len > p.code.size()) return -1;
    const uint32_t op = ins.x & 0xFF;
    pc += len;
    if (op == OP_NOP) continue;
    if (ins.x & F_NARROW) { if (!narrow_step(ins, &p.code[pc - len + 1])) return -1; continue; }
    if (op == OP_SPILL_ST) { if (ins.y >= p.n_regs || ins.z >= p.n_spill) return -1; spill[ins.z] = rf[ins.y]; continue; }
    if (op == OP_POW5) {
      const uint32_t reg = ins.y & 0xFFFF, d4 = ins.y >> 16;
      if (reg >= p.n_regs) return -1;
      const fe x2 = fe_sqr(rf[reg]), x4 = fe_sqr(x2), x5 = fe_mul(x4, rf[reg]);
      if (ins.z != NO_POS) { if (ins.z >= p.n_witness) return -1; memcpy(witness + 32 * (size_t)ins.z, x2.l, 32); }
      if (d4 != 0xFFFF) { if (ins.z == NO_POS || ins.z + d4 >= p.n_witness) return -1; memcpy(witness + 32 * (size_t)(ins.z + d4), x4.l, 32); }
      if (!commit(ins, x5)) return -1;
      continue;
    }
    fe R;
    if (!compute(ins, &p.code[pc - len + 1], &R) || !commit(ins, R)) return -1;
  }
  return st;
}
// inputs JSON -> I x 32 B buffer; returns 0 ok / 1 error (message in err)
int sim_inputs(SimGraph* s, const char* json, uint8_t* buf, char* err, size_t errlen) {
  try {
    InputList in = deserialize_inputs(json, strlen(json));
    std::vector<U256> b = build_inputs_buffer(s->g, in);
    memcpy(buf, b.data(), b.size() * 32);
    return 0;
  } catch (const std::exception& e) { if (err && errlen) { strncpy(err, e.what(), errlen - 1); err[errlen - 1] = 0; } return 1; }
}
// re-serialise the parsed graph (codec round trip); returns the size, copies up to cap bytes
size_t sim_reserialize(SimGraph* s, uint8_t* out, size_t cap) {
  std::vector<uint8_t> v = serialize_witnesscalc_graph(s->g);
  if (out && cap >= v.size()) memcpy(out, v.data(), v.size());
  return v.size();
}
void sim_wtns_header(uint32_t n, uint8_t* dst) { wtns_write_header(dst, n); }

// latency plan (plan.hpp: LatencyPlan): the main warps run level by level; inside a level every instruction reads
// its operands before ANY instruction of the level writes (the kernel runs them concurrently), which exposes slot
// hazards.  The slow warps are asynchronous on the device; the simulator runs each job at one of the two extremes
// the protocol allows -- mode 0: as soon as its issue level starts, mode 1: just before the OP_WAIT that guards its
// readers -- so a slot recycled too early (or a reader scheduled before the wait) shows up as a wrong witness.
// opts (11 words): {n_warps, n_slow_warps, slow_levels, split_dot, fuse, packet_slots, chain, dataflow, sbox_links (2 = forced),
// exclusive_warp0, max_slots} (0 = default for the counts and sizes)
// out10: n_levels, n_slots, n_instrs, max level width, status, est_cycles, n_split | n_rows, slow_levels, n_chained | n_waits, n_sbox_links
// cov (LAT_COV_WORDS words or null): what the kernel would execute, accumulated over calls (LatCov below)
enum LatCov {
  COV_DOT_SHAPES,     // mask of the straight-line OP_DOT shapes executed (bit = ins.y >> 16)
  COV_DOT_TERMS,      // largest term count of a generic-loop OP_DOT
  COV_DOT_KINDS,      // mask of the term kinds of generic-loop OP_DOTs (bit = T_*)
  COV_SLOW_WIDTHS,    // mask of the lanes of slow-warp jobs (bit = headers of the job, 1..32)
  COV_SLOW_OPS,       // mask of the opcodes of slow-warp jobs
  COV_SLOW_CONST,     // slow-warp instructions that read a constant operand
  COV_POW5, COV_POW4, COV_MULADD, COV_SHRAND, COV_OUT, COV_TERN_CONST, COV_MULADD_CONST,
  COV_CHAIN,          // largest number of headers per lane in one packet
  COV_LEVELS_MOD3,    // mask of n_levels mod 3
  COV_LEVELS_SMALL,   // mask of n_levels below 64
  COV_EMPTY_PACKET,   // level plan: packets of a main warp without headers
  COV_CHUNK_FULL,     // dataflow plan: chunks filled to their last slot
  COV_CHUNK_ZERO,     // dataflow plan: chunks ended by a zero descriptor
  COV_WAIT_WIDTH,     // dataflow plan: largest number of nonzero entries of a wait vector
  COV_PHYS_WARPS,     // dataflow plan: n_phys_warps
  COV_N_SLOTS, COV_MAX_SLOTS,
  COV_DOT_SHAPES_M1,  // mask of the straight-line OP_DOT shapes executed with a first-product constant of M - 1 (worst case)
  LAT_COV_WORDS
};
int64_t sim_eval_latency3(SimGraph* s, const uint8_t* inputs, uint8_t* witness, uint64_t* out8, int mode, const uint32_t* opts, uint64_t* cov) {
  const std::vector<uint32_t> key(opts, opts + 11);
  if (!s->lat_ok || s->lat_key != key) {
    s->lat_ok = false;
    try {
      LatencyOptions o;
      if (opts[0]) o.n_warps = opts[0]; if (opts[1]) o.n_slow_warps = opts[1]; o.slow_levels = opts[2]; o.split_dot = opts[3] != 0; o.fuse = opts[4] != 0; if (opts[5]) o.packet_slots = opts[5]; o.chain = opts[6] != 0; o.dataflow = opts[7] != 0; o.sbox_links = opts[8] != 0; o.force_sbox_links = opts[8] == 2;
      o.exclusive_warp0 = opts[9] != 0; if (opts[10]) o.max_slots = opts[10];
      s->lat = compile_latency_plan(s->g, o);
      s->lat_key = key; s->lat_ok = true;
    } catch (const std::exception& e) { s->err = e.what(); return -2; }
  }
  const LatencyPlan& lp = s->lat;
  uint64_t dummy[LAT_COV_WORDS] = {};
  uint64_t* cv = cov ? cov : dummy;
  cv[COV_LEVELS_MOD3] |= 1ull << (lp.n_levels % 3);
  if (lp.n_levels < 64) cv[COV_LEVELS_SMALL] |= 1ull << lp.n_levels;
  cv[COV_N_SLOTS] = std::max<uint64_t>(cv[COV_N_SLOTS], lp.n_slots);
  cv[COV_MAX_SLOTS] = opts[10] ? opts[10] : LatencyOptions().max_slots;
  if (lp.dataflow) cv[COV_PHYS_WARPS] = std::max<uint64_t>(cv[COV_PHYS_WARPS], lp.n_phys_warps);
  // what one header makes the kernel do (lat_exec; lat_exec_slow for the jobs of the slow warps)
  auto cover = [&](size_t pk, const Instr& ins, bool slow) {
    const uint32_t op = ins.x & 0xFF;
    const bool any_const = (ins.x & F_A_CONST) || ((ins.x & F_B_CONST) && op_has_b_host(op)) || ((ins.x & F_C_CONST) && (op == OP_TERN || op == OP_MULADD));
    if (op == OP_NOP) return;
    if (slow) { cv[COV_SLOW_OPS] |= 1ull << op; cv[COV_SLOW_CONST] += any_const; }
    if (op == OP_DOT) {
      const uint32_t nt = ins.y & 0xFF, shape = ins.y >> 16;
      if (shape & 1) {
        cv[COV_DOT_SHAPES] |= 1ull << shape;
        const fe m1 = fe_neg(fe_small(1));
        const size_t ci = pk + ins.z < lp.code.size() ? pk + lp.code[pk + ins.z].y : lp.code.size();
        if (ci + 1 < lp.code.size()) {
          const Instr& a = lp.code[ci]; const Instr& b = lp.code[ci + 1];
          const uint32_t v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
          if (!memcmp(v, m1.l, 32)) cv[COV_DOT_SHAPES_M1] |= 1ull << shape;
        }
      } else {
        cv[COV_DOT_TERMS] = std::max<uint64_t>(cv[COV_DOT_TERMS], nt);
        for (uint32_t t = 0; t < nt && pk + ins.z + (t >> 1) < lp.code.size(); t++) {
          const Instr& sl = lp.code[pk + ins.z + (t >> 1)];
          cv[COV_DOT_KINDS] |= 1ull << (((t & 1) ? sl.z : sl.x) & 0xF);
        }
      }
    }
    cv[COV_POW5] += op == OP_POW5; cv[COV_POW4] += op == OP_POW4; cv[COV_MULADD] += op == OP_MULADD; cv[COV_SHRAND] += op == OP_SHRAND;
    cv[COV_OUT] += op == OP_OUT; cv[COV_TERN_CONST] += op == OP_TERN && any_const; cv[COV_MULADD_CONST] += op == OP_MULADD && any_const;
  };
  auto cover_packet = [&](size_t pk, uint32_t nh, uint32_t lanes, bool slow) {
    if (lanes) cv[COV_CHAIN] = std::max<uint64_t>(cv[COV_CHAIN], (nh + lanes - 1) / lanes);
    if (slow) cv[COV_SLOW_WIDTHS] |= 1ull << nh;
    for (uint32_t k = 0; k < nh && pk + 1 + k < lp.code.size(); k++) cover(pk, lp.code[pk + 1 + k], slow);
  };
  std::vector<fe> slots(lp.n_slots, fe_zero());
  uint32_t st = 0;
  struct W { uint32_t dst; fe v; };
  // operands: a slot of the value file, or a constant stored inline in the packet (two slots at a packet-relative offset)
  auto pconst = [&](size_t pk, uint32_t rel, fe* o) {
    if (pk + rel + 1 >= lp.code.size()) return false;
    const Instr& a = lp.code[pk + rel]; const Instr& b = lp.code[pk + rel + 1];
    o->l[0] = a.x; o->l[1] = a.y; o->l[2] = a.z; o->l[3] = a.w; o->l[4] = b.x; o->l[5] = b.y; o->l[6] = b.z; o->l[7] = b.w;
    return true;
  };
  // a lane sees its own earlier writes of the level (program order); everybody else's only after the level barrier
  std::map<uint32_t, fe> overlay;
  auto rslot = [&](uint32_t idx) { auto it = overlay.find(idx); return it != overlay.end() ? it->second : slots[idx]; };
  auto load = [&](size_t pk, uint32_t idx, bool is_const, fe* o) { if (is_const) return pconst(pk, idx, o); if (idx >= lp.n_slots) return false; *o = rslot(idx); return true; };
  // value of one header of the packet at `pk` from the current slot file; writes go to `writes`
  auto exec = [&](size_t pk, const Instr& ins, std::vector<W>& writes) {
    const uint32_t op = ins.x & 0xFF, dst = ins.x >> 16;
    if (op == OP_NOP) return true;
    fe A = fe_zero(), B = fe_zero(), C = fe_zero(), R;
    if (op == OP_INPUT) { if (ins.y >= lp.n_inputs) return false; fe v; memcpy(v.l, inputs + 32 * (size_t)ins.y, 32); R = fe_reduce256(v); }
    else if (op == OP_DOT) {
      const uint32_t nt = ins.y & 0xFF, ncs = (ins.y >> 8) & 0xFF;
      if (nt == 0 || nt > DOT_MAX_TERMS || ncs < 1 || ncs > 3 || pk + ins.z + ((nt + 1) >> 1) > lp.code.size()) return false;
      dot_acc P; dot_init(P);
      for (uint32_t t = 0; t < nt; t++) {
        const Instr& sl = lp.code[pk + ins.z + (t >> 1)];
        const uint32_t lo = (t & 1) ? sl.z : sl.x, ci = (t & 1) ? sl.w : sl.y;
        const uint32_t kind = lo & 0xF, reg = lo >> 16;
        fe c = fe_zero();
        if (kind > T_CONST || reg >= lp.n_slots) return false;
        if ((kind == T_MAC || kind == T_CONST) && !pconst(pk, ci, &c)) return false;
        dot_term(P, kind, rslot(reg), c);
      }
      R = fe_mont_reduce(P, (int)ncs);
    } else if (op == OP_POW5) {
      const uint32_t reg = ins.y & 0xFFFF, d4 = ins.y >> 16;
      if (reg >= lp.n_slots) return false;
      const fe x = rslot(reg), x2 = fe_sqr(x), x4 = fe_sqr(x2);
      if (ins.z != NO_POS) { if (ins.z >= lp.n_witness) return false; memcpy(witness + 32 * (size_t)ins.z, x2.l, 32); }
      if (d4 != 0xFFFF) { if (ins.z == NO_POS || ins.z + d4 >= lp.n_witness) return false; memcpy(witness + 32 * (size_t)(ins.z + d4), x4.l, 32); }
      R = fe_mul(x4, x);
    } else if (op == OP_POW4) {
      if (ins.y >= lp.n_slots) return false;
      const fe x2 = fe_sqr(rslot(ins.y));
      if (ins.z != NO_POS) { if (ins.z >= lp.n_witness) return false; memcpy(witness + 32 * (size_t)ins.z, x2.l, 32); }
      R = fe_sqr(x2);
    } else if (op == OP_MULADD) {
      if (!load(pk, ins.y, ins.x & F_A_CONST, &A) || !load(pk, ins.z, ins.x & F_B_CONST, &B) || !load(pk, ins.w, ins.x & F_C_CONST, &C)) return false;
      R = fe_add(fe_mul(A, B), C);
    } else if (op == OP_SHRAND) {
      fe c;
      if (ins.y >= lp.n_slots || !pconst(pk, ins.z >> 8, &c)) return false;
      R = fe_shr_and(rslot(ins.y), ins.z & 0xFF, c);
    } else {
      if (!load(pk, ins.y, ins.x & F_A_CONST, &A)) return false;
      if (op == OP_OUT) { if (ins.w >= lp.n_witness) return false; memcpy(witness + 32 * (size_t)ins.w, A.l, 32); return true; }
      if (op_has_b(op) && !load(pk, ins.z, ins.x & F_B_CONST, &B)) return false;
      if (op == OP_TERN && !load(pk, ins.w, ins.x & F_C_CONST, &C)) return false;
      R = alu_exec(op, A, B, C, st);
    }
    if (dst != NO_DST) { if (dst >= lp.n_slots) return false; writes.push_back({dst, R}); overlay[dst] = R; }
    if ((ins.x & F_OUT) && op != OP_TERN && op != OP_MULADD) { if (ins.w >= lp.n_witness) return false; memcpy(witness + 32 * (size_t)ins.w, R.l, 32); }
    return true;
  };
  if (lp.dataflow) {
    // Dataflow plan: every warp walks its own stream; a packet may start when the progress counters of the other warps
    // have reached its wait vector.  The simulator picks the next runnable warp by policy -- mode 0: lowest warp first
    // (slow warps as late as possible), mode 1: highest warp first (slow warps as early as possible), mode >= 2: pseudo-
    // random with seed `mode` -- so that a missing wait (operand not yet produced, slot overwritten before its last
    // reader) shows up as a wrong witness, and a cyclic wait as a deadlock (-4).
    const uint32_t NW = lp.n_phys_warps, C = lp.chunk_slots;
    if (lp.stream_off.size() != NW || C == 0) return -1;
    std::vector<uint32_t> progress(NW, 0), chunk(NW, 0), off(NW, 0);
    uint64_t rng = 0x9E3779B97F4A7C15ull * (uint64_t)(mode + 1), n_headers = 0;
    auto cursor = [&](uint32_t w, size_t* pk) {            // next packet of warp w, or false at the end of its stream
      while (chunk[w] < lp.stream_chunks[w]) {
        const size_t base = (size_t)lp.stream_off[w] + (size_t)chunk[w] * C;
        if (off[w] < C && lp.code[base + off[w]].x != 0) { *pk = base + off[w]; return true; }
        if (off[w] >= C) cv[COV_CHUNK_FULL]++; else cv[COV_CHUNK_ZERO]++;
        chunk[w]++; off[w] = 0;
      }
      return false;
    };
    auto runnable = [&](uint32_t w, size_t pk) {
      const Instr& d = lp.code[pk];
      if (!d.z) return true;
      for (uint32_t x = 0; x < NW; x++) {
        const Instr& sl = lp.code[pk + d.z + x / 4];
        const uint32_t need = (x & 3) == 0 ? sl.x : (x & 3) == 1 ? sl.y : (x & 3) == 2 ? sl.z : sl.w;
        if (x != w && progress[x] < need) return false;
      }
      return true;
    };
    for (;;) {
      std::vector<uint32_t> cand;
      bool any_left = false;
      for (uint32_t w = 0; w < NW; w++) { size_t pk; if (cursor(w, &pk)) { any_left = true; if (runnable(w, pk)) cand.push_back(w); } }
      if (!any_left) break;
      if (cand.empty()) return -4;
      uint32_t w;
      if (mode == 0) w = cand.front(); else if (mode == 1) w = cand.back();
      else { rng ^= rng << 13; rng ^= rng >> 7; rng ^= rng << 17; w = cand[(size_t)(rng % cand.size())]; }
      size_t pk; cursor(w, &pk);
      const Instr d = lp.code[pk];
      const uint32_t nh = d.y & 0xFFFFu, lanes = d.y >> 16;
      if (d.x > C - off[w] || nh + 1 > d.x || lanes > 32 || (nh && !lanes) || d.w != progress[w] + 1) return -1;
      if (d.z) {
        uint64_t nz = 0;
        for (uint32_t x = 0; x < NW; x++) { const Instr& sl = lp.code[pk + d.z + x / 4]; nz += ((x & 3) == 0 ? sl.x : (x & 3) == 1 ? sl.y : (x & 3) == 2 ? sl.z : sl.w) != 0; }
        cv[COV_WAIT_WIDTH] = std::max(cv[COV_WAIT_WIDTH], nz);
      }
      cover_packet(pk, nh, lanes, nh && lat_is_slow_op(lp.code[pk + 1].x & 0xFF));
      std::vector<W> writes;
      for (uint32_t lane = 0; lane < lanes; lane++) {
        overlay.clear();
        for (uint32_t k = lane; k < nh; k += lanes) { if (!exec(pk, lp.code[pk + 1 + k], writes)) return -1; n_headers++; }
      }
      overlay.clear();
      for (const W& x : writes) slots[x.dst] = x.v;
      progress[w] = d.w;
      off[w] += d.x;
    }
    out8[0] = lp.n_levels; out8[1] = lp.n_slots; out8[2] = lp.n_instrs; out8[3] = lp.max_level_width; out8[4] = st;
    out8[5] = lp.est_cycles; out8[6] = lp.n_rows; out8[7] = lp.slow_levels; out8[8] = lp.n_waits_df; out8[9] = lp.n_sbox_links;
    return 0;
  }
  std::vector<uint32_t> next_job(lp.n_slow_warps, 0);
  auto run_job = [&](uint32_t w, uint32_t j) {
    const uint32_t* e = &lp.jobs[((size_t)w * lp.max_jobs + j) * 4];
    if ((size_t)e[1] + e[2] >= lp.code.size()) return false;
    cover_packet(e[1], e[2], e[2], true);
    std::vector<W> writes;
    for (uint32_t k = 0; k < e[2]; k++) { overlay.clear(); if ((size_t)e[1] + 1 + k >= lp.code.size() || !exec(e[1], lp.code[e[1] + 1 + k], writes)) return false; }
    overlay.clear();
    for (const W& x : writes) slots[x.dst] = x.v;
    return true;
  };
  // packets of the main warps: levels 0 and 1 from `first`, level L + 2 from the descriptor of level L (what the kernel walks)
  std::vector<uint32_t> cur(lp.n_warps * 4), nxt(lp.n_warps * 4);
  for (uint32_t w = 0; w < lp.n_warps; w++) for (int k = 0; k < 4; k++) { cur[w * 4 + k] = lp.first[w * 8 + k]; nxt[w * 4 + k] = lp.first[w * 8 + 4 + k]; }
  uint64_t n_headers = 0;
  size_t next_wait = 0;
  for (uint32_t L = 0; L < lp.n_levels; L++) {
    for (uint32_t w = 0; w < lp.n_warps; w++) if ((size_t)cur[w * 4] + cur[w * 4 + 1] > lp.code.size() || cur[w * 4 + 2] + 1 > cur[w * 4 + 1] || cur[w * 4 + 3] > 32 || (cur[w * 4 + 2] && !cur[w * 4 + 3])) return -1;
    // slow jobs first: mode 0 = every job issued at this level, mode 1 = the jobs this level's OP_WAITs wait for
    if (mode == 0) {
      for (uint32_t w = 0; w < lp.n_slow_warps; w++)
        while (next_job[w] < lp.n_jobs[w] && lp.jobs[((size_t)w * lp.max_jobs + next_job[w]) * 4] <= L) { if (!run_job(w, next_job[w])) return -1; next_job[w]++; }
    } else {
      for (; next_wait * 4 < lp.waits.size() && lp.waits[next_wait * 4] == L; next_wait++) {
        const uint32_t ws = lp.waits[next_wait * 4 + 1], seq = lp.waits[next_wait * 4 + 2];
        if (ws >= lp.n_slow_warps || seq > lp.n_jobs[ws]) return -1;
        while (next_job[ws] < seq) {
          if (lp.jobs[((size_t)ws * lp.max_jobs + next_job[ws]) * 4] > L) return -3;     // waits for a job that cannot have started
          if (!run_job(ws, next_job[ws])) return -1;
          next_job[ws]++;
        }
      }
    }
    std::vector<W> writes;
    for (uint32_t w = 0; w < lp.n_warps; w++) {
      const size_t pk = cur[w * 4];
      const uint32_t nh = cur[w * 4 + 2], lanes = cur[w * 4 + 3];
      if (nh == 0) cv[COV_EMPTY_PACKET]++;
      cover_packet(pk, nh, lanes, false);
      for (uint32_t lane = 0; lane < lanes; lane++) {
        overlay.clear();
        for (uint32_t k = lane; k < nh; k += lanes) { if (!exec(pk, lp.code[pk + 1 + k], writes)) return -1; n_headers++; }
      }
    }
    overlay.clear();
    for (const W& x : writes) slots[x.dst] = x.v;
    for (uint32_t w = 0; w < lp.n_warps; w++) {
      const Instr d = lp.code[cur[w * 4]];
      for (int k = 0; k < 4; k++) cur[w * 4 + k] = nxt[w * 4 + k];
      nxt[w * 4] = d.x; nxt[w * 4 + 1] = d.y; nxt[w * 4 + 2] = d.z; nxt[w * 4 + 3] = d.w;
    }
  }
  for (uint32_t w = 0; w < lp.n_slow_warps; w++) while (next_job[w] < lp.n_jobs[w]) { if (!run_job(w, next_job[w])) return -1; next_job[w]++; }
  out8[0] = lp.n_levels; out8[1] = lp.n_slots; out8[2] = lp.n_instrs; out8[3] = lp.max_level_width; out8[4] = st;
  out8[5] = lp.est_cycles; out8[6] = lp.n_split; out8[7] = lp.slow_levels; out8[8] = lp.n_chained; out8[9] = lp.n_sbox_links;
  return 0;
}
int64_t sim_eval_latency2(SimGraph* s, const uint8_t* inputs, uint8_t* witness, uint64_t* out8, int mode, const uint32_t* opts) {
  uint32_t o[11] = {0, 0, 0, 1, 1, 0, 1, 0, 1, 0, 0};
  if (opts) for (int k = 0; k < 9; k++) o[k] = opts[k];
  return sim_eval_latency3(s, inputs, witness, out8, mode, o, nullptr);
}
const char* sim_error(SimGraph* s) { return s->err.c_str(); }
int64_t sim_eval_latency(SimGraph* s, const uint8_t* inputs, uint8_t* witness, uint64_t* out5) {
  uint64_t o8[10];
  int64_t rc = sim_eval_latency2(s, inputs, witness, o8, 0, nullptr);
  if (rc == 0) for (int k = 0; k < 5; k++) out5[k] = o8[k];
  return rc;
}
}

// ---- bit-sliced plan (bitplan.hpp) on the host: one group of up to 32 input sets, exactly what bit_eval_kernel and
// bit_expand_kernel do (contract check + pack, steps of 32 LUTs on one word per plane, expansion of the plane words) ----
#include "../../circom-witnesscalc_b200/csrc/bitplan.hpp"

struct BitSim { Graph g; BitPlan bp; };

extern "C" {

BitSim* sim_bit_load2(const uint8_t* data, size_t len, uint32_t max_support, int merge, uint32_t max_slots, char* err, size_t errlen);
BitSim* sim_bit_load(const uint8_t* data, size_t len, uint32_t max_support, int merge, char* err, size_t errlen) {
  return sim_bit_load2(data, len, max_support, merge, 0, err, errlen);
}
// max_slots: GW_BIT_MAX_SLOTS (0 = default)
BitSim* sim_bit_load2(const uint8_t* data, size_t len, uint32_t max_support, int merge, uint32_t max_slots, char* err, size_t errlen) {
  try {
    std::unique_ptr<BitSim> s(new BitSim());
    s->g = deserialize_witnesscalc_graph(data, len);
    BitPlanOptions o; if (max_support) o.max_support = max_support; o.merge_luts = merge != 0; if (max_slots) o.max_slots = max_slots;
    s->bp = compile_bit_plan(s->g, o);
    if (!s->bp.eligible && err && errlen) { strncpy(err, s->bp.reason.c_str(), errlen - 1); err[errlen - 1] = 0; }
    return s.release();
  } catch (const std::exception& e) { if (err && errlen) { strncpy(err, e.what(), errlen - 1); err[errlen - 1] = 0; } return nullptr; }
}
void sim_bit_free(BitSim* s) { delete s; }
void sim_bit_info(BitSim* s, uint64_t* out) {
  const BitPlan& b = s->bp;
  out[0] = b.eligible; out[1] = b.n_steps; out[2] = b.n_slots; out[3] = b.n_luts; out[4] = b.n_levels; out[5] = b.n_nodes_bit;
  out[6] = b.n_nodes_tt; out[7] = b.n_nodes_bv; out[8] = b.n_full_adders; out[9] = b.n_merged; out[10] = b.inputs.size() / 3; out[11] = b.const_vals.size();
  out[12] = b.has_field_inputs; out[13] = b.wide.size() / 3; out[14] = b.plane_stride;
}
// the compiled plan: which = 0 code (4 words per LUT), 1 inputs (triples), 2 wide (triples), 3 const_of_pos (int32 as
// uint32); copies up to cap words and returns the number of words
size_t sim_bit_plan(BitSim* s, int which, uint32_t* out, size_t cap) {
  const BitPlan& b = s->bp;
  const uint32_t* src = which == 0 ? reinterpret_cast<const uint32_t*>(b.code.data()) : which == 1 ? b.inputs.data() : which == 2 ? b.wide.data() : (const uint32_t*)b.const_of_pos.data();
  const size_t n = which == 0 ? b.code.size() * 4 : which == 1 ? b.inputs.size() : which == 2 ? b.wide.size() : b.const_of_pos.size();
  if (out && src) memcpy(out, src, std::min(n, cap) * 4);
  return n;
}
// inputs: n x I x 32 B (n <= 32), witness: n x W x 32 B; returns the mask of input sets that satisfy the bit contract
// (only their rows are written), or -1 on a malformed plan
int64_t sim_bit_eval(BitSim* s, const uint8_t* inputs, uint32_t n, uint8_t* witness) {
  const BitPlan& b = s->bp;
  if (!b.eligible || n > 32) return -1;
  std::vector<uint32_t> S(b.n_slots, 0);
  S[BIT_SLOT_ONES] = 0xFFFFFFFFu;
  uint32_t ok = n == 32 ? 0xFFFFFFFFu : ((1u << n) - 1);
  for (size_t k = 0; k + 2 < b.inputs.size() + 0 && k < b.inputs.size(); k += 3) {
    const uint32_t idx = b.inputs[k], slot = b.inputs[k + 1], bit = b.inputs[k + 2];
    if (idx >= b.n_inputs) return -1;
    uint32_t word = 0;
    for (uint32_t w = 0; w < n; w++) {
      const uint8_t* v = inputs + ((size_t)w * b.n_inputs + idx) * 32;
      if (bit == BIT_CONTRACT) {
        bool is_bit = v[0] <= 1;
        for (int q = 1; q < 32; q++) is_bit &= v[q] == 0;
        if (!is_bit) ok &= ~(1u << w);
        word |= (uint32_t)(v[0] & 1) << w;
      } else {
        if (bit >= 254) return -1;
        fe x; memcpy(x.l, v, 32);
        x = fe_reduce256(x);                                     // Fr::new (graph.rs:376)
        word |= ((x.l[bit >> 5] >> (bit & 31)) & 1u) << w;
      }
    }
    if (slot != BIT_NO_SLOT) { if (slot >= b.n_slots) return -1; S[slot] = word; }
  }
  if (b.plane_stride < b.n_witness) return -1;
  std::vector<uint32_t> planes(b.plane_stride, 0);
  for (uint32_t st = 0; st < b.n_steps; st++) {
    uint32_t res[32]; 
    for (uint32_t lane = 0; lane < 32; lane++) {                 // all lanes read ...
      const BitOp& op = b.code[(size_t)st * 32 + lane];
      const uint32_t sa = op.y & 0xFFFF, sb = op.y >> 16, sc = op.z & 0xFFFF;
      if (sa >= b.n_slots || sb >= b.n_slots || sc >= b.n_slots) return -1;
      res[lane] = bit_lut3(op.x & 0xFF, S[sa], S[sb], S[sc]);
    }
    for (uint32_t lane = 0; lane < 32; lane++) {                 // ... before any lane writes
      const BitOp& op = b.code[(size_t)st * 32 + lane];
      const uint32_t dst = op.z >> 16;
      if (dst != BIT_NO_SLOT) { if (dst >= b.n_slots || dst < 2) return -1; S[dst] = res[lane]; }
      if (op.w != BIT_NO_POS) { if (op.w >= b.plane_stride) return -1; planes[op.w] = res[lane]; }
    }
  }
  for (uint32_t w = 0; w < n; w++) {
    if (!((ok >> w) & 1)) continue;
    for (uint32_t j = 0; j < b.n_witness; j++) {
      uint8_t* dst = witness + ((size_t)w * b.n_witness + j) * 32;
      if (b.const_of_pos[j] >= 0) memcpy(dst, b.const_vals[(size_t)b.const_of_pos[j]].l, 32);
      else if (b.const_of_pos[j] == -1) { memset(dst, 0, 32); dst[0] = (planes[j] >> w) & 1; }
    }
    for (size_t q = 0; q + 2 < b.wide.size() + 0 && q < b.wide.size(); q += 3) {
      const uint32_t pos = b.wide[q], base = b.wide[q + 1], np = b.wide[q + 2];
      if (pos >= b.n_witness || np > 256 || b.n_witness + base + np > b.plane_stride) return -1;
      uint8_t* dst = witness + ((size_t)w * b.n_witness + pos) * 32;
      memset(dst, 0, 32);
      for (uint32_t p = 0; p < np; p++) dst[p >> 3] |= (uint8_t)(((planes[b.n_witness + base + p] >> w) & 1u) << (p & 7));
    }
  }
  return (int64_t)ok;
}

}  // extern "C"
