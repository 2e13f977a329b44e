// Graph -> device program ("plan").
//
// This is the load-time half of what replaces /root/reference/src/graph.rs:367-391 (evaluate): the
// reference walks Vec<Node> and keeps one Fr per node (N x 32 B per witness).  For a batch that does
// not fit (authV2: 194 k nodes -> 6 MB per witness), so the node list is compiled once into a linear
// instruction stream over a small per-witness register file (shared memory on the device) with
// Belady-style spilling to a witness-major spill area in HBM.  Dead nodes are dropped, constants go
// to a deduplicated table, witness positions are attached to the defining instruction.
//
// Two graph-level rewrites run first (both preserve every node value bit for bit):
//   * Div batching: Div nodes on the same "division level" are independent, so groups of up to
//     `div_batch` of them share ONE modular inversion (Montgomery's trick: 4k-3 multiplications + 1
//     inversion instead of k inversions), with b == 0 -> 0 kept exact (graph.rs:109).
//   * Linear-combination fusion: trees of Add/Sub whose inner nodes are single-use temporaries and whose
//     leaves are Mul(value, constant) become one OP_DOT: products are accumulated in 512 bits and
//     reduced once (the reference's build-circuit emits `lc += c * x` chains, SURVEY Appendix A).
#pragma once
#include "graph.hpp"
#include "isa.h"

namespace gw {

struct PlanOptions {
  uint32_t n_regs = 12;      // per-witness registers kept in shared memory (12 x 32 B x 512 threads = 192 KB)
  uint32_t div_batch = 8;    // max Div nodes sharing one inversion (1 = off)
  bool fuse_dot = true;      // fuse linear combinations into OP_DOT
  uint32_t max_terms = 8;    // max terms of one OP_DOT (<= DOT_MAX_TERMS, <= n_regs - 3)
  bool narrow = true;        // narrow typing: provably small values are computed on int64 (isa.h: F_NARROW)
  bool fuse_pow5 = true;     // Sqr -> Sqr -> Mul S-box chains become one OP_POW5 (throughput plan)
  bool fold_addc = false;    // Mul(constant, value +- constant) -> OP_DOT terms that do not wait for the Add (latency mode)
};

struct PlanStats {
  uint64_t graph_nodes = 0, graph_ops = 0;   // ops = Op + UnoOp + TresOp nodes of the file (node-ops/s metric)
  uint64_t live_ops = 0;                     // ops of the file reachable from the witness
  uint64_t instrs = 0, slots = 0, spill_st = 0, spill_ld = 0, outs = 0;
  uint64_t op_count[64] = {0};               // emitted instructions by opcode
  uint64_t dot_terms[4] = {0, 0, 0, 0};      // emitted OP_DOT terms by TermKind
  uint64_t inversions = 0;                   // modular inversions per witness (OP_DIV + OP_INV)
  uint64_t div_nodes = 0;                    // live Div nodes of the graph
  uint64_t mul_nodes = 0;                    // live Mul nodes of the graph
  uint32_t max_live = 0;                     // peak number of simultaneously live values
  uint64_t narrow_instrs = 0;                // emitted narrow (int64) instructions, spill moves excluded
  uint64_t pow5 = 0;                         // S-box chains fused into OP_POW5
};

struct Plan {
  std::vector<Instr> code;   // slots
  std::vector<U256> consts;
  uint32_t n_regs = 0, n_spill = 0;
  uint32_t n_spill_narrow = 0;   // 8-byte spill slots of narrow values (a pool of their own: [slot][thread] uint2)
  uint32_t n_inputs = 0;     // I: length of the input buffer incl. slot 0
  uint32_t n_witness = 0;    // W
  PlanStats stats;
};

Plan compile_plan(const Graph& g, const PlanOptions& opt);

// c * 2^256 mod M (or (M - c) * 2^256 mod M): the form OP_DOT constants are stored in (c canonical)
U256 prescale(const U256& c, bool neg);

// Single-witness ("latency") mode.  The macro ops (fused linear combinations included) are scheduled level by
// level: all instructions of a level are independent.  A level's instructions are spread over `n_warps` MAIN
// warps of one CTA -- instructions of the same class share a warp (SIMT lanes), different classes go to different
// warps (different SM sub-partitions) -- and a named barrier over the main warps separates levels.  The long
// operations (Div/Inv/Pow/Idiv/Mod: tens of thousands of cycles) do not hold a level up: they are queued, in groups
// of up to 32 of the same opcode, to `n_slow_warps` SLOW warps that run asynchronously; a job starts when the main
// warps have published the level that produces its operands and its readers are scheduled `slow_levels` levels
// later, behind a wait on the job's completion counter that a CONTROL warp performs before it joins the barrier of
// the level in front of them (the control warp also publishes the completed levels: it has no asynchronous copies
// in flight, so its fences are cheap).  Operands name slots of one shared-memory value file;
// a slot is recycled only at a level boundary after its last reader (for a slow reader: after the level at which the control warp waits for it).
//
//   code   : packets.  A packet is what ONE warp needs for ONE level (or one slow-warp job), contiguous: slot 0 =
//            descriptor {offset, slots, headers, lanes of the same warp's packet two levels later}, then the headers
//            (header k belongs to lane k mod lanes; a lane runs its headers in order: a chain), then
//            what the headers point at with packet-relative slot offsets: OP_DOT tails (.z) and every constant operand
//            (two slots each; OP_DOT terms carry the offset of their constant) -- one asynchronous global->shared
//            copy brings a level's instructions and constants on chip, with no register in flight across a barrier.
//   first  : [n_warps][2] {offset, slots, headers, lanes} of the packets of levels 0 and 1
//   jobs   : [n_slow_warps][max_jobs] {issue level, packet offset, number of headers, 0}
//   waits  : {level, slow warp, number of jobs of that warp that must be complete before the level ends, 0}
struct LatencyOptions {
  uint32_t max_slots = 7000;     // capacity of the shared-memory value file (32 B slots)
  uint32_t packet_slots = 128;   // capacity of one stage of the kernel's packet ring (16 B slots): wide levels are cut to fit
  uint32_t n_warps = 7;          // main warps that execute instructions (one more warp publishes levels and waits for jobs)
  uint32_t n_slow_warps = 4;
  uint32_t slow_levels = 0;      // levels between the issue of a long op and its first reader; 0 = from the cost model
  bool split_dot = true;         // split a linear combination into an early part (operands known early) and a late part
  bool fuse = true;              // OP_DOT / OP_SHRAND fusion (off: one instruction per graph node)
  bool chain = true;             // run single-reader chains (x^2 -> x^4 -> x^5) in one lane inside one level
  uint32_t max_chain = 4;        // instructions per chain
  bool force_sbox_links = false; // apply the rewrite below whatever the timing model says (tests)
  bool sbox_links = true;        // S*x^5 on the path from one S-box to the next becomes (S*x)*x^4: OP_POW4 + OP_MULADD (plan.cpp: rewrite_sbox_links)
  bool dataflow = false;         // per-warp packet streams with wait vectors instead of level barriers (eval_dataflow_kernel)
  bool exclusive_warp0 = false;  // dataflow: warp 0 takes the critical instructions and shares its SM sub-partition with nobody (measured: no gain)
};
struct LatencyPlan {
  std::vector<Instr> code;
  std::vector<uint32_t> first;        // 8 words per main warp
  std::vector<uint32_t> jobs;         // 4 words per (slow warp, job)
  std::vector<uint32_t> n_jobs;       // per slow warp
  std::vector<uint32_t> waits;        // 4 words per wait, ascending levels: {level, slow warp, jobs that must be complete, 0}
  uint32_t n_levels = 0, n_warps = 0, n_slow_warps = 0, max_jobs = 0, slow_levels = 0;
  uint32_t n_slots = 0, n_inputs = 0, n_witness = 0;
  uint32_t max_level_width = 0;
  uint64_t n_instrs = 0, n_slow = 0, n_split = 0, n_chained = 0;
  uint64_t est_cycles = 0;            // cost model: sum over levels of the slowest warp + per-level overhead
  // dataflow plan (LatencyOptions::dataflow): code = the streams of warps 0 .. n_warps + n_slow_warps - 1, each a whole
  // number of chunks of chunk_slots slots.  A chunk holds packets back to back: slot 0 of a packet = {slots of the packet
  // (0: the chunk ends here), headers | lanes << 16, packet-relative slot of its wait vector (0: none), the packet's
  // 1-based number in its warp's stream}; headers and extras as in a level-plan packet; the wait vector is 12 words:
  // how many packets of warp k must be complete before this one starts.
  bool dataflow = false;
  std::vector<uint32_t> stream_off, stream_chunks;
  uint32_t chunk_slots = 0, n_phys_warps = 0;     // stream_off / stream_chunks have n_phys_warps entries (some may be empty)
  uint64_t n_rows = 0, n_waits_df = 0;
  uint64_t n_sbox_links = 0;          // S-box to S-box links rewritten (LatencyOptions::sbox_links)
};
LatencyPlan compile_latency_plan(const Graph& g, const LatencyOptions& opt);

}  // namespace gw
