// Batch witness evaluator for sm_100a: the device half of what replaces
// /root/reference/src/graph.rs:367-391 (graph::evaluate).
//
// Execution model (throughput mode): one thread = one input set ("witness").  All 32 lanes of a
// warp run the SAME instruction of the plan for 32 different witnesses, so opcode dispatch is
// warp-uniform and there is no divergence.  Each warp streams the 16-byte instructions itself:
// lane l loads instruction base+l (one coalesced 512 B read), the next block of 32 is prefetched
// while the current one executes, and the instruction being executed is broadcast with shuffles, so
// warps never synchronise with each other.  Values live in a per-witness register file in shared
// memory laid out [register][half][thread] as uint4 (conflict-free LDS.128/STS.128); values that do
// not fit are spilled to HBM witness-major ([slot][half][thread], coalesced 128-bit accesses).
// Witness values are written canonical, 32 B each, at witness[w][position].
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <memory>
#include <mutex>
#include <vector>

#include "engine.hpp"
#include "alu.cuh"
#include "cuda_util.hpp"

namespace gw {

struct KParams {
  const uint4* code; uint32_t n_slots;
  const uint4* consts; uint32_t n_hot;   // the first n_hot table constants (most used first) are staged in shared memory
  const uint4* inputs;     // [B][I][2]
  uint4* out;              // [B][W][2]
  uint4* spill;            // [n_spill][2][spill_threads]
  uint2* nspill;           // [n_spill_narrow][spill_threads]: narrow values (threads of different warps are at
                           // different instructions, so a slot must never change its per-thread layout)
  uint32_t* status;        // [B] or null
  unsigned long long B;
  uint32_t I, W;
  uint32_t n_tiles;
  unsigned long long spill_threads;
  // optional indirection (the bit-sliced path's fallback): evaluate the input sets row_map[0 .. *n_dev) instead of 0 .. B
  const uint32_t* row_map; const uint32_t* n_dev;
#ifdef GW_PROFILING
  unsigned long long out_wrap;   // profiling aid (GW_DEBUG_OUT_WRAP, -DGW_PROFILING builds only): witness rows wrap modulo this many rows; 0 = off
#endif
};

__device__ __forceinline__ fe fe_from(uint4 lo, uint4 hi) {
  fe r; r.l[0] = lo.x; r.l[1] = lo.y; r.l[2] = lo.z; r.l[3] = lo.w; r.l[4] = hi.x; r.l[5] = hi.y; r.l[6] = hi.z; r.l[7] = hi.w; return r;
}
__device__ __forceinline__ uint4 fe_lo(const fe& a) { return make_uint4(a.l[0], a.l[1], a.l[2], a.l[3]); }
__device__ __forceinline__ uint4 fe_hi(const fe& a) { return make_uint4(a.l[4], a.l[5], a.l[6], a.l[7]); }
__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }

static const int RING = 64;          // instruction slots staged per warp in shared memory (two blocks of 32)
#ifndef GW_MAX_THREADS
#define GW_MAX_THREADS 512           // one persistent CTA per SM; 512 threads x 128 registers = the whole register file
#endif
static const int MAX_THREADS = GW_MAX_THREADS;

// One thread = one input set; blockDim.x = T threads (a multiple of 32, chosen per launch so that one CTA per SM covers
// the batch).  Dynamic shared memory: [T/32 warps][RING] instruction slots | [n_hot][2] hot constants | register file
// [n_regs][2 halves][T], all uint4.  Warps never synchronise with each other after the constants are staged.
__global__ void __launch_bounds__(MAX_THREADS, 1) eval_batch_kernel(const KParams p) {
  extern __shared__ uint4 smem[];
  const int T = blockDim.x;
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  uint4* ring = smem + (tid >> 5) * RING;
  uint4* hot = smem + (T >> 5) * RING;
  uint4* rf = hot + 2 * (size_t)p.n_hot + tid;       // this thread's column of the register file
  const unsigned long long gthread = (unsigned long long)blockIdx.x * T + tid;
  const uint32_t n = p.n_slots;
  const unsigned long long B = p.n_dev ? (unsigned long long)*p.n_dev : p.B;       // uniform over the grid
  const uint32_t n_tiles = p.n_dev ? (uint32_t)((B + T - 1) / T) : p.n_tiles;
  if (blockIdx.x >= n_tiles) return;

  for (uint32_t k = tid; k < 2 * p.n_hot; k += T) hot[k] = __ldg(p.consts + k);
  __syncthreads();

  auto rf_load = [&](uint32_t r) { return fe_from(rf[(r * 2) * T], rf[(r * 2 + 1) * T]); };
  auto rf_store = [&](uint32_t r, const fe& x) { rf[(r * 2) * T] = fe_lo(x); rf[(r * 2 + 1) * T] = fe_hi(x); };
  auto const_load = [&](uint32_t c) {
    if (c < p.n_hot) return fe_from(hot[2 * c], hot[2 * c + 1]);
    return fe_from(__ldg(p.consts + 2 * (size_t)c), __ldg(p.consts + 2 * (size_t)c + 1));
  };
  // narrow values: limbs 0..1 only
  auto nrf_load2 = [&](uint32_t r) { return *reinterpret_cast<const uint2*>(&rf[(r * 2) * T]); };
  auto nrf_load = [&](uint32_t r) { const uint2 v = nrf_load2(r); return (int64_t)((uint64_t)v.x | ((uint64_t)v.y << 32)); };
  auto nrf_store = [&](uint32_t r, int64_t x) { *reinterpret_cast<uint2*>(&rf[(r * 2) * T]) = make_uint2((uint32_t)(uint64_t)x, (uint32_t)((uint64_t)x >> 32)); };
  auto nconst_load = [&](uint32_t c) {
    const uint2 v = (c < p.n_hot) ? *reinterpret_cast<const uint2*>(&hot[2 * c]) : __ldg(reinterpret_cast<const uint2*>(p.consts + 2 * (size_t)c));
    return (int64_t)((uint64_t)v.x | ((uint64_t)v.y << 32));
  };

  for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const unsigned long long w = (unsigned long long)tile * T + tid;
    const bool active = w < B;
    const unsigned long long wi = active ? w : B - 1;
    const unsigned long long wl = p.row_map ? (unsigned long long)p.row_map[wi] : wi;     // row of the input / witness arrays
    const uint4* in = p.inputs + wl * p.I * 2;
#ifdef GW_PROFILING
    uint4* out = p.out + (p.out_wrap ? wl % p.out_wrap : wl) * p.W * 2;
#else
    uint4* out = p.out + wl * p.W * 2;
#endif
    uint32_t st = 0;
    auto out_store = [&](uint32_t j, const fe& x) { if (active) { out[2 * (size_t)j] = fe_lo(x); out[2 * (size_t)j + 1] = fe_hi(x); } };

    // instruction ring: blocks 0 and 1 staged, block 2 in flight in nblk
    __syncwarp();
    ring[lane] = __ldg(p.code + min((uint32_t)lane, n - 1));
    ring[32 + lane] = __ldg(p.code + min(32u + lane, n - 1));
    uint4 nblk = __ldg(p.code + min(64u + lane, n - 1));
    __syncwarp();
    uint32_t pc = 0;
    uint4 nxt = ring[0];
    while (pc < n) {
      const uint4 ins = nxt;
      const uint32_t op = ins.x & 0xFFu;
      const uint32_t dst = ins.x >> 16;
      const uint32_t len = (op == OP_DOT) ? 1u + (((ins.y & 0xFFu) + 1u) >> 1) : 1u;
      const uint32_t npc = pc + len;
      const bool cross = (npc >> 5) != (pc >> 5);
      if (!cross) nxt = ring[npc & (RING - 1)];     // next header early: its latency hides behind this instruction

      fe R;
      bool have_result = true;
      if (ins.x & F_NARROW) {
        // narrow instruction (isa.h): int64 values in limbs 0..1 of their registers, 8-byte moves
        int64_t r = 0;
        bool have_r = true;
        if (op == OP_DOT) {
          const uint32_t nt = ins.y & 0xFFu;
#pragma unroll 1
          for (uint32_t t = 0; t < nt; t++) {
            const uint4 sl = ring[(pc + 1 + (t >> 1)) & (RING - 1)];
            const uint32_t lo = (t & 1) ? sl.z : sl.x, ci = (t & 1) ? sl.w : sl.y;
            const uint32_t kind = lo & 0xFu;
            const int64_t x = (kind == T_CONST) ? 0 : nrf_load(lo >> 16);
            const int64_t c = (kind == T_MAC || kind == T_CONST) ? nconst_load(ci) : 0;
            r = narrow_dot_term(r, kind, x, c);
          }
        } else if (op == OP_SPILL_ST) {
          p.nspill[(size_t)ins.z * p.spill_threads + gthread] = nrf_load2(ins.y);
          have_r = false;
        } else if (op == OP_SPILL_LD) {
          const uint2 v = p.nspill[(size_t)ins.y * p.spill_threads + gthread];
          r = (int64_t)((uint64_t)v.x | ((uint64_t)v.y << 32));
        } else if (op == OP_OUT) {
          out_store(ins.w, fe_from_narrow(nrf_load(ins.y)));
          have_r = false;
        } else if (op == OP_SHRAND) {
          r = narrow_shr_and(nrf_load(ins.y), ins.z & 0xFFu, nconst_load(ins.z >> 8));
        } else {
          const int64_t a = (ins.x & F_A_CONST) ? nconst_load(ins.y) : nrf_load(ins.y);
          int64_t b = 0, c = 0;
          if (op_has_b(op)) b = (ins.x & F_B_CONST) ? nconst_load(ins.z) : nrf_load(ins.z);
          if (op == OP_TERN) c = (ins.x & F_C_CONST) ? nconst_load(ins.w) : nrf_load(ins.w);
          r = narrow_exec(op, a, b, c);
        }
        if (have_r) {
          if (dst != NO_DST) nrf_store(dst, r);
          if (ins.x & F_OUT) out_store(ins.w, fe_from_narrow(r));
        }
        have_result = false;
      } else if (op == OP_DOT) {
        // fused linear combination: 512-bit accumulator, ONE Montgomery reduction
        const uint32_t nt = ins.y & 0xFFu;
        dot_acc P;
        dot_init(P);
#pragma unroll 1
        for (uint32_t t = 0; t < nt; t++) {
          const uint4 sl = ring[(pc + 1 + (t >> 1)) & (RING - 1)];
          const uint32_t lo = (t & 1) ? sl.z : sl.x, ci = (t & 1) ? sl.w : sl.y;
          const uint32_t kind = lo & 0xFu, reg = lo >> 16;
          if (kind == T_MAC) {
            const fe c = const_load(ci);
            const fe x = rf_load(reg);
            dot_mac(P, x.l, c.l);
          } else if (kind == T_CONST) {
            const fe c = const_load(ci);
            dot_add256(P, c.l, 0);
          } else {
            dot_term(P, kind, rf_load(reg), fe_zero());
          }
        }
        R = fe_mont_reduce(P, (int)((ins.y >> 8) & 0xFFu));
      } else if (op == OP_MUL || op == OP_SQR) {
        const fe A = (ins.x & F_A_CONST) ? const_load(ins.y) : rf_load(ins.y);
        uint32_t Pm[16];
        if (op == OP_SQR) {
          u256_sqr_wide(Pm, A.l);
        } else {
          const fe Bv = (ins.x & F_B_CONST) ? const_load(ins.z) : rf_load(ins.z);
          u256_mul_wide(Pm, A.l, Bv.l);
        }
        R = fe_barrett(Pm);
      } else if (op == OP_POW5) {
        // Poseidon S-box in one instruction: x^2 and x^4 go straight to their witness positions (isa.h)
        const fe A = rf_load(ins.y & 0xFFFFu);
        const uint32_t d4 = ins.y >> 16;
        uint32_t Pm[16];
        u256_sqr_wide(Pm, A.l);
        const fe x2 = fe_barrett(Pm);
        if (ins.z != NO_POS) out_store(ins.z, x2);
        u256_sqr_wide(Pm, x2.l);
        const fe x4 = fe_barrett(Pm);
        if (d4 != 0xFFFFu) out_store(ins.z + d4, x4);
        u256_mul_wide(Pm, x4.l, A.l);
        R = fe_barrett(Pm);
      } else if (op == OP_ADD || op == OP_SUB) {
        const fe A = (ins.x & F_A_CONST) ? const_load(ins.y) : rf_load(ins.y);
        const fe Bv = (ins.x & F_B_CONST) ? const_load(ins.z) : rf_load(ins.z);
        R = (op == OP_ADD) ? fe_add(A, Bv) : fe_sub(A, Bv);
      } else if (op == OP_SPILL_ST) {
        const fe x = rf_load(ins.y);
        p.spill[((size_t)ins.z * 2) * p.spill_threads + gthread] = fe_lo(x);
        p.spill[((size_t)ins.z * 2 + 1) * p.spill_threads + gthread] = fe_hi(x);
        have_result = false;
      } else if (op == OP_SPILL_LD) {
        R = fe_from(p.spill[((size_t)ins.y * 2) * p.spill_threads + gthread], p.spill[((size_t)ins.y * 2 + 1) * p.spill_threads + gthread]);
      } else if (op == OP_OUT) {
        out_store(ins.w, (ins.x & F_A_CONST) ? const_load(ins.y) : rf_load(ins.y));
        have_result = false;
      } else if (op == OP_INPUT) {
        R = fe_reduce256(fe_from(__ldg(in + 2 * (size_t)ins.y), __ldg(in + 2 * (size_t)ins.y + 1)));
      } else if (op == OP_SHRAND) {
        R = fe_shr_and(rf_load(ins.y), ins.z & 0xFFu, const_load(ins.z >> 8));
      } else if (op != OP_NOP) {
        // everything else (Div, Inv and the rare ops; out-of-line helpers)
        const fe A = (ins.x & F_A_CONST) ? const_load(ins.y) : rf_load(ins.y);
        fe Bv = fe_zero(), C = fe_zero();
        if (op_has_b(op)) Bv = (ins.x & F_B_CONST) ? const_load(ins.z) : rf_load(ins.z);
        if (op == OP_TERN) C = (ins.x & F_C_CONST) ? const_load(ins.w) : rf_load(ins.w);
        R = alu_exec(op, A, Bv, C, st);
      } else {
        have_result = false;
      }
      if (have_result) {
        if (dst != NO_DST) rf_store(dst, R);
        if (ins.x & F_OUT) out_store(ins.w, R);
      }

      if (cross) {
        // block (pc >> 5) is consumed: stage block (pc >> 5) + 2 in its half, start loading the one after it
        __syncwarp();
        ring[((pc >> 5) & 1u) * 32u + lane] = nblk;
        nblk = __ldg(p.code + min(((pc >> 5) + 3u) * 32u + lane, n - 1));
        __syncwarp();
        nxt = ring[npc & (RING - 1)];
      }
      pc = npc;
    }
    if (p.status != nullptr && active) p.status[wl] = st;
  }
}

// ---- bit-sliced path for Boolean graphs (bitplan.hpp) ---------------------------------------------------------------
// One warp = one GROUP of 32 input sets.  A plane is one 32-bit word of the warp's plane file in shared memory: bit k =
// the value for input set 32 g + k.  The plan is a sequence of steps of 32 independent 3-input look-up tables; in a step
// every LANE executes its own LUT (lane = instruction, word = 32 input sets), so a step costs one coalesced 512-byte
// header load, three shared-memory reads, ~25 logic instructions and one write per lane, and warps never synchronise
// with each other.  The prologue packs the inputs into planes and CHECKS the contract the plan was typed under (every
// input is 0 or 1); input sets that break it are handed to eval_batch_kernel through bad_list.
struct BParams {
  const uint4* code; uint32_t n_steps, n_slots;
  uint32_t warp_bytes;                      // shared memory per warp: plane file (+ mbarriers + header ring), a multiple of 16
  const uint4* in_list; uint32_t n_in;      // {input index, plane slot or BIT_NO_SLOT, bit or BIT_CONTRACT, 0}: contract inputs first, then the bits of field inputs
  uint32_t n_contract;                      // the first n_contract entries of in_list are the contract inputs (batch kernels: the rest comes from the tables below)
  const uint32_t* field_inputs; uint32_t n_field;   // input indices of the field inputs
  const uint32_t* field_slots;              // [n_field][256]: plane slot of bit b of field input f, or BIT_NO_SLOT
  const uint4* inputs;                      // [B][I][2]
  uint32_t I, W;
  unsigned long long B;
  uint32_t n_groups;
  uint32_t* planes; uint32_t plane_stride;  // [n_groups][plane_stride]: plane word of every witness position, then the planes of the wide values
  uint32_t* ok_words;                       // [n_groups]: bit k = input set 32 g + k satisfies the contract
  uint32_t* bad_list; uint32_t* n_bad;      // the other input sets, for the fallback launch
  uint32_t* status;                         // [B] or null (per-set flags: 0 for every set evaluated here)
};

static const uint32_t BIT_PREFETCH = 4;
static const uint32_t BIT_CHUNK_SINGLE = 16, BIT_CHUNK_BATCH = 8;      // steps per TMA chunk of a warp's header ring (3 stages)

__device__ __forceinline__ uint32_t lut3_eval(uint32_t lut, uint32_t a, uint32_t b, uint32_t c) {
  // branch-free (the 32 lanes hold 32 different tables): a multiplexer tree over the 8 table bits spread to masks
#define GW_LM(k) ((uint32_t)((int32_t)(lut << (31 - (k))) >> 31))
  const uint32_t t0 = (a & GW_LM(1)) | (~a & GW_LM(0));
  const uint32_t t1 = (a & GW_LM(3)) | (~a & GW_LM(2));
  const uint32_t t2 = (a & GW_LM(5)) | (~a & GW_LM(4));
  const uint32_t t3 = (a & GW_LM(7)) | (~a & GW_LM(6));
#undef GW_LM
  const uint32_t u0 = (b & t1) | (~b & t0), u1 = (b & t3) | (~b & t2);
  return (c & u1) | (~c & u0);
}

// SINGLE: one input set (the single-witness entry points): only bit 0 of a plane word means anything, so a LUT is one
// table look-up (5 dependent instructions instead of the 3-level multiplexer tree) -- the step loop of one warp is a
// pure latency chain: shared-memory read, LUT, write, __syncwarp.
// RING: the LUT headers of a warp come through its own 3-stage shared-memory ring filled by TMA bulk copies (CH steps per
// chunk) instead of register prefetches: a warp's step is a dependent chain of ~100-200 cycles, an L2 round trip for the
// header is longer than that, and ptxas batches register prefetches at the end of the unrolled body.  Costs shared
// memory (fewer resident groups per SM), so large batches may prefer the register variant (launch_bit).
template <bool SINGLE, bool RING>
__global__ void __launch_bounds__(256) bit_eval_kernel(const BParams p) {
  extern __shared__ uint32_t bit_smem[];
  // (SINGLE: one warp.  Saying so keeps every address below provably warp-uniform: with `threadIdx.x >> 5` in them the
  // compiler guards each __syncwarp of the step loop with a divergence check -- 0.45 -> 0.62 ms on SHA-256, measured)
  const uint32_t lane = threadIdx.x & 31u, warp = SINGLE ? 0u : __shfl_sync(0xFFFFFFFFu, threadIdx.x >> 5, 0);   // a shuffle from lane 0: warp-uniform for the compiler too
  const uint32_t g = blockIdx.x * (blockDim.x >> 5) + warp;
  if (g >= p.n_groups) return;
  uint32_t* S = bit_smem + (size_t)warp * (p.warp_bytes >> 2);          // [plane file][3 mbarriers][ring] per warp
  const unsigned long long row = (unsigned long long)g * 32u + lane;
  const bool in_range = row < p.B;
  if (lane == 0) { S[BIT_SLOT_ZERO] = 0u; S[BIT_SLOT_ONES] = 0xFFFFFFFFu; }
  // pack + contract check: lane = input set.  A contract input must be 0 or 1 and is its own plane; of a field input
  // (taken apart by the graph with Shr/Band) the planes are bits of the value reduced mod M, whatever the value.
  const uint4* in = p.inputs + (in_range ? row : 0ull) * p.I * 2;
  bool ok = in_range;
  if (SINGLE) {
    // one input set: lane = entry of the input list (32 entries per pass instead of one dependent L2 round trip each)
    ok = true;
    for (uint32_t k0 = 0; k0 < p.n_in; k0 += 32u) {
      const uint32_t k = k0 + lane;
      if (k < p.n_in) {
        const uint4 e = __ldg(p.in_list + k);
        const uint4 lo = __ldg(p.inputs + 2 * (size_t)e.x), hi = __ldg(p.inputs + 2 * (size_t)e.x + 1);
        if (e.z == BIT_CONTRACT) {
          ok = ok && (lo.x <= 1u) && ((lo.y | lo.z | lo.w | hi.x | hi.y | hi.z | hi.w) == 0u);
          if (e.y != BIT_NO_SLOT) S[e.y] = lo.x & 1u;
        } else {
          const fe w = fe_reduce256(fe_from(lo, hi));
          uint32_t limb = 0;
#pragma unroll
          for (uint32_t q = 0; q < 8; q++) limb = (q == (e.z >> 5)) ? w.l[q] : limb;
          S[e.y] = (limb >> (e.z & 31u)) & 1u;
        }
      }
    }
    ok = __all_sync(0xFFFFFFFFu, ok) && lane == 0;        // lane 0 stands for the input set below
  } else {
    // contract inputs: 32 list entries per coalesced load, then one ballot per entry
    for (uint32_t k0 = 0; k0 < p.n_contract; k0 += 32u) {
      const uint4 mine = (k0 + lane < p.n_contract) ? __ldg(p.in_list + k0 + lane) : make_uint4(0, BIT_NO_SLOT, 0, 0);
      const uint32_t n = min(32u, p.n_contract - k0);
      for (uint32_t k = 0; k < n; k++) {
        const uint32_t ex = __shfl_sync(0xFFFFFFFFu, mine.x, k), ey = __shfl_sync(0xFFFFFFFFu, mine.y, k);
        const uint4 lo = __ldg(in + 2 * (size_t)ex), hi = __ldg(in + 2 * (size_t)ex + 1);
        ok = ok && (lo.x <= 1u) && ((lo.y | lo.z | lo.w | hi.x | hi.y | hi.z | hi.w) == 0u);
        const uint32_t word = __ballot_sync(0xFFFFFFFFu, in_range && (lo.x & 1u));
        if (lane == 0 && ey != BIT_NO_SLOT) S[ey] = word;
      }
    }
    // field inputs (Fr::new, graph.rs:376: the planes are bits of the canonical value): a 32 x 32 bit transpose across
    // the warp per limb -- lane j ends up with the plane word of bit 32 q + j -- instead of one ballot per bit
    for (uint32_t f = 0; f < p.n_field; f++) {
      const uint32_t ix = __ldg(p.field_inputs + f);
      const fe w = fe_reduce256(fe_from(__ldg(in + 2 * (size_t)ix), __ldg(in + 2 * (size_t)ix + 1)));
#pragma unroll
      for (uint32_t q = 0; q < 8; q++) {
        uint32_t x = in_range ? w.l[q] : 0u;
#pragma unroll
        for (uint32_t j = 16; j >= 1; j >>= 1) {
          const uint32_t m = j == 16 ? 0x0000FFFFu : j == 8 ? 0x00FF00FFu : j == 4 ? 0x0F0F0F0Fu : j == 2 ? 0x33333333u : 0x55555555u;
          const uint32_t y = __shfl_xor_sync(0xFFFFFFFFu, x, j);
          x = (lane & j) ? (((y >> j) & m) | (x & (m << j))) : ((x & m) | ((y & m) << j));
        }
        const uint32_t slot = __ldg(p.field_slots + f * 256u + q * 32u + lane);
        if (slot != BIT_NO_SLOT) S[slot] = x;
      }
    }
  }
  const uint32_t okw = __ballot_sync(0xFFFFFFFFu, ok);
  if (lane == 0) p.ok_words[g] = okw;
  if (in_range && !ok) p.bad_list[atomicAdd(p.n_bad, 1u)] = (uint32_t)row;
  if (p.status != nullptr && ok) p.status[row] = 0u;
  if (okw == 0u) return;                                   // nobody in this group honours the contract
  __syncwarp();
  uint32_t* planes = p.planes + (size_t)g * p.plane_stride;
  // the headers of the next BIT_PREFETCH steps are in flight while a step executes: one L2 round trip per step would
  // otherwise be the whole cost of a step (a handful of warps per SM cannot hide it)
  if (RING) {
    // chunk c + 2 is requested when chunk c starts; a chunk completes on the mbarrier of its stage
    constexpr uint32_t BIT_CHUNK = SINGLE ? BIT_CHUNK_SINGLE : BIT_CHUNK_BATCH;
    const uint32_t smem_s = (uint32_t)__cvta_generic_to_shared(S);
    const uint32_t bar_s = smem_s + ((p.n_slots * 4u + 15u) & ~15u), ring_s = bar_s + 32u;
    const uint32_t n_chunks = (p.n_steps - 1u + BIT_CHUNK - 1u) / BIT_CHUNK;     // steps 1 .. n_steps - 1
    if (lane < 3u) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_s + 8u * lane) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncwarp();
    auto request = [&](uint32_t c) {
      if (c >= n_chunks || lane != 0u) return;
      const uint32_t stage = c % 3u, first = 1u + c * BIT_CHUNK;
      const uint32_t bytes = min(BIT_CHUNK, p.n_steps - first) * 512u, bar = bar_s + 8u * stage;
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");          // earlier generic reads of the stage vs the async write
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"(ring_s + stage * (BIT_CHUNK * 512u)), "l"(p.code + (size_t)first * 32u), "r"(bytes), "r"(bar) : "memory");
    };
    request(0); request(1);
    for (uint32_t c = 0; c < n_chunks; c++) {
      const uint32_t stage = c % 3u, parity = (c / 3u) & 1u, bar = bar_s + 8u * stage;
      uint32_t done = 0;
      while (!done)
        asm volatile("{ .reg .pred q; mbarrier.try_wait.parity.shared::cta.b64 q, [%1], %2; selp.u32 %0, 1, 0, q; }" : "=r"(done) : "r"(bar), "r"(parity) : "memory");
      __syncwarp();                                                         // every lane is done with chunk c - 1: its stage may be refilled
      request(c + 2u);
      const uint32_t n = min(BIT_CHUNK, p.n_steps - 1u - c * BIT_CHUNK);
      const uint32_t src = ring_s + stage * (BIT_CHUNK * 512u) + lane * 16u;
      uint4 nxt;
      asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(nxt.x), "=r"(nxt.y), "=r"(nxt.z), "=r"(nxt.w) : "r"(src));
      for (uint32_t k = 0; k < n; k++) {
        const uint4 ins = nxt;
        if (k + 1u < n) asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(nxt.x), "=r"(nxt.y), "=r"(nxt.z), "=r"(nxt.w) : "r"(src + (k + 1u) * 512u));
        const uint32_t a = S[ins.y & 0xFFFFu], b = S[ins.y >> 16], cc = S[ins.z & 0xFFFFu];
        const uint32_t r = SINGLE ? ((ins.x >> ((a & 1u) | ((b & 1u) << 1) | ((cc & 1u) << 2))) & 1u) : lut3_eval(ins.x, a, b, cc);
        const uint32_t dst = ins.z >> 16;
        if (dst != BIT_NO_SLOT) S[dst] = r;
        if (ins.w != BIT_NO_POS) planes[ins.w] = r;
        __syncwarp();
      }
    }
    return;
  }
  const uint32_t last = p.n_steps - 1u;
  constexpr uint32_t PF = BIT_PREFETCH;
  uint4 q[PF];
#pragma unroll
  for (uint32_t k = 0; k < PF; k++) q[k] = __ldg(p.code + (size_t)min(1u + k, last) * 32u + lane);   // step 0 is the prologue above
  for (uint32_t st = 1; st < p.n_steps; st += PF) {
#pragma unroll
    for (uint32_t k = 0; k < PF; k++) {
      const uint4 ins = q[k];
      q[k] = __ldg(p.code + (size_t)min(st + k + PF, last) * 32u + lane);
      if (st + k < p.n_steps) {                              // uniform
        const uint32_t a = S[ins.y & 0xFFFFu], b = S[ins.y >> 16], c = S[ins.z & 0xFFFFu];
        const uint32_t r = lut3_eval(ins.x, a, b, c);
        const uint32_t dst = ins.z >> 16;
        if (dst != BIT_NO_SLOT) S[dst] = r;                  // never a slot another lane reads in this step (bitplan.cpp)
        if (ins.w != BIT_NO_POS) planes[ins.w] = r;
        __syncwarp();
      }
    }
  }
}

// Plane words -> canonical 32-byte witness values.  A warp takes one group and 32 consecutive witness positions (one
// plane word per lane) and writes, for each of the group's input sets, the 32 x 32 bytes of that stretch of the set's
// witness row with two 512-byte coalesced streaming stores: the HBM-bound part of the bit-sliced path.
__global__ void __launch_bounds__(256) bit_expand_kernel(const uint32_t* __restrict__ planes, const uint32_t* __restrict__ ok_words,
                                                         const int32_t* __restrict__ const_of_pos, const uint4* __restrict__ consts,
                                                         uint4* __restrict__ out, uint32_t W, uint32_t plane_stride, uint32_t n_groups,
                                                         uint32_t tiles_per_group) {
  const uint32_t lane = threadIdx.x & 31u;
  const unsigned long long t = (unsigned long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const uint32_t g = (uint32_t)(t / tiles_per_group);
  if (g >= n_groups) return;
  const uint32_t j0 = (uint32_t)(t % tiles_per_group) * 32u, j = j0 + lane;
  const uint32_t okw = __ldg(ok_words + g);
  if (okw == 0u) return;
  const int32_t cidx = j < W ? __ldg(const_of_pos + j) : -1;
  const uint32_t word = (j < W && cidx == -1) ? __ldg(planes + (size_t)g * plane_stride + j) : 0u;   // constants and wide values have no plane
  const uint32_t half = lane & 1u;
  for (uint32_t w = 0; w < 32u; w++) {
    if (!((okw >> w) & 1u)) continue;
    uint4* row = out + ((size_t)g * 32u + w) * W * 2;
#pragma unroll
    for (uint32_t h = 0; h < 2u; h++) {
      const uint32_t pz = h * 16u + (lane >> 1);
      const uint32_t wv = __shfl_sync(0xFFFFFFFFu, word, pz);
      const int32_t ci = __shfl_sync(0xFFFFFFFFu, cidx, pz);
      if (j0 + pz < W && ci != -2) {                           // -2: a wide value, written by bit_expand_wide_kernel
        uint4 v = make_uint4(half ? 0u : ((wv >> w) & 1u), 0u, 0u, 0u);
        if (ci >= 0) v = __ldg(consts + 2 * (size_t)ci + half);
        __stcs(row + 2 * (size_t)(j0 + pz) + half, v);
      }
    }
  }
}

// Witness values that are integers of several bits (Bits2Num sums, field inputs passed through): one warp per (group,
// wide value) transposes up to 256 planes into the 8 limbs of each of the group's 32 input sets.
__global__ void __launch_bounds__(256) bit_expand_wide_kernel(const uint32_t* __restrict__ planes, const uint32_t* __restrict__ ok_words,
                                                              const uint4* __restrict__ wide, uint32_t n_wide, uint32_t* __restrict__ out,
                                                              uint32_t W, uint32_t plane_stride, uint32_t n_groups) {
  const uint32_t lane = threadIdx.x & 31u;
  const unsigned long long t = (unsigned long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const uint32_t g = (uint32_t)(t / n_wide);
  if (g >= n_groups) return;
  const uint4 d = __ldg(wide + (uint32_t)(t % n_wide));      // {position, base, number of planes, 0}
  const uint32_t okw = __ldg(ok_words + g);
  if (okw == 0u) return;
  const uint32_t* src = planes + (size_t)g * plane_stride + W + d.y;
  uint32_t P[8];
#pragma unroll
  for (uint32_t m = 0; m < 8; m++) P[m] = (32u * m + lane < d.z) ? __ldg(src + 32u * m + lane) : 0u;
  for (uint32_t w = 0; w < 32u; w++) {
    if (!((okw >> w) & 1u)) continue;
    uint32_t mine = 0;
#pragma unroll
    for (uint32_t m = 0; m < 8; m++) {
      const uint32_t limb = __ballot_sync(0xFFFFFFFFu, (P[m] >> w) & 1u);
      mine = lane == m ? limb : mine;
    }
    if (lane < 8u) out[(((size_t)g * 32u + w) * W + d.x) * 8u + lane] = mine;
  }
}

// ---- single-witness latency mode ------------------------------------------------------------------------
// One CTA evaluates ONE witness (plan.hpp: LatencyPlan).  MAIN warps run the plan level by level: every lane takes
// one instruction (or one chain of instructions) of the level -- instructions of one class share a warp, different
// classes sit in different warps and therefore on different SM sub-partitions -- values live in one shared-memory slot
// file, a named barrier over the main warps and the control warp separates levels.  SLOW warps run the long operations
// (Div/Inv/Pow/Idiv/Mod) asynchronously: a job starts when the level that produces its operands has been published,
// and the CONTROL warp waits for the job counter of that slow warp before it joins the barrier in front of the job's
// readers.  The control warp also feeds the main warps: the packet (headers, OP_DOT tails, constants) of level L+2
// lands in a 3-stage shared-memory ring per main warp by TMA while level L executes.
struct LParams {
  const uint4* code; const uint4* first; uint32_t n_levels, n_warps;
  const uint4* jobs; const uint32_t* n_jobs; uint32_t max_jobs, n_slow;
  const uint4* waits; uint32_t n_waits;
  const uint4* inputs;     // [I][2]
  uint4* out;              // [W][2]
  uint32_t* status;        // [1] or null
  uint32_t n_slots;
  uint32_t dbg;            // GW_LAT_DBG, timing experiments only: 1 = no witness stores, 16 = no instructions (level skeleton alone)
  unsigned long long* level_clock;   // profiling aid (GW_LAT_CLOCKS): clock64 at the end of every level, or null
  // batch form (BATCH = true): CTA b evaluates input set row_map ? row_map[b] : b; inputs [.][I][2], out [.][W][2], status [.]
  const uint32_t* row_map; uint32_t I, W;
};

static const int LAT_MAX_THREADS = 384;     // main + control + slow warps <= 12: 170 registers per thread
static const uint32_t LAT_RING_SLOTS = 128; // packet ring: 3 stages x 2 KB per main warp (plan.hpp: LatencyOptions::packet_slots)
static const uint32_t LAT_CTRL_BYTES = 320; // 32 B control words (levels, job counters) + 3 mbarriers x up to 11 main warps, 16 B aligned

// Shared memory is addressed with 32-bit shared-window addresses and explicit ld/st.shared: a generic pointer costs a
// window lookup (S2R) per access in this kernel's dependent chains.
__device__ __forceinline__ uint4 lds128(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t a, const uint4 v) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ fe lds_fe(uint32_t a) { return fe_from(lds128(a), lds128(a + 16)); }
// Progress flags between warps that do not share a barrier (completed levels, jobs done per slow warp): written and
// polled with shared-memory atomics by ONE lane (an atomic is never a data race, and 32 lanes hammering one word would
// serialise); the block-level fences around them order the value-file accesses they publish.
__device__ __forceinline__ void flag_publish(uint32_t a, uint32_t v) {
  __threadfence_block();
  asm volatile("{ .reg .b32 old; atom.shared.exch.b32 old, [%0], %1; }" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t flag_read(uint32_t a) {
  uint32_t v;
  asm volatile("atom.shared.or.b32 %0, [%1], 0;" : "=r"(v) : "r"(a) : "memory");
  return v;
}
// The barrier that ends a level: main warps and the control warp arrive at ONE barrier instruction (a function of its
// own, so that every participant executes the same bar.sync: what compute-sanitizer's synccheck expects of an aligned barrier).
__device__ __noinline__ void lat_level_barrier(uint32_t n_threads) { asm volatile("bar.sync 1, %0;" ::"r"(n_threads) : "memory"); }
// the whole warp waits until the flag at shared address a reaches v
__device__ __forceinline__ void flag_wait(uint32_t a, uint32_t v, uint32_t lane, uint32_t sleep_ns) {
  if (lane == 0) while (flag_read(a) < v) __nanosleep(sleep_ns);
  __syncwarp();
  __threadfence_block();
}

// The rare operations live in one out-of-line function so that the code a main warp walks every level (Mul, Sqr,
// OP_DOT, Add/Sub, stores) stays small; the slow warps call nothing else.
__device__ __noinline__ void lat_exec_rare(uint32_t op, const fe& A, const fe& Bv, const fe& C, uint32_t* st, fe* R) {
  uint32_t s = 0;
  *R = alu_exec(op, A, Bv, C, s);
  *st |= s;
}
struct LatCtx {
  const uint4* inputs; uint4* out;
  uint32_t slots_s;        // shared-window address of the value file
  uint32_t dbg;
};
// one instruction of the packet at shared address pk_s (a stage of the warp's packet ring)
__device__ __forceinline__ void lat_exec(const LatCtx& cx, uint32_t pk_s, const uint4 ins, uint32_t* st) {
  auto slot_load = [&](uint32_t r) { return lds_fe(cx.slots_s + 32u * r); };
  auto const_load = [&](uint32_t rel) { return lds_fe(pk_s + 16u * rel); };
  auto operand = [&](uint32_t is_const, uint32_t idx) { return is_const ? const_load(idx) : slot_load(idx); };
  const uint32_t op = ins.x & 0xFFu, dst = ins.x >> 16;
  fe R;
  if (op == OP_NOP) return;
  if (op == OP_OUT) { fe v = operand(ins.x & F_A_CONST, ins.y); cx.out[2 * (size_t)ins.w] = fe_lo(v); cx.out[2 * (size_t)ins.w + 1] = fe_hi(v); return; }
  if (op == OP_DOT) {
    const uint32_t nt = ins.y & 0xFFu;
    const uint32_t tail_s = pk_s + 16u * ins.z;
    const uint32_t shape = ins.y >> 16;
    dot_acc P;
    dot_init(P);
    if (shape & 1u) {
      // straight-line path for the Poseidon mix shapes (plan.cpp: shape hint): every operand fetch is issued up front,
      // no term loop, no per-term dispatch
      const uint32_t n_mac = (shape >> 1) & 3u;
      const uint4 t01 = lds128(tail_s), t23 = lds128(tail_s + 16u);
      const fe x0 = slot_load(t01.x >> 16), c0 = const_load(t01.y);
      // term 1 is the second product, or the added value, or the constant; term 2 / 3 follow in that order
      uint32_t k = 1;
      fe x1 = x0, c1 = c0;
      if (n_mac == 2) { x1 = slot_load(t01.z >> 16); c1 = const_load(t01.w); k = 2; }
      fe av = x0, cv = c0;
      if (shape & 8u) { av = slot_load((k == 1 ? t01.z : t23.x) >> 16); k++; }
      if (shape & 16u) cv = const_load(k == 1 ? t01.w : k == 2 ? t23.y : t23.w);
      dot_mac(P, x0.l, c0.l);
      if (n_mac == 2) dot_mac(P, x1.l, c1.l);
      if (shape & 8u) dot_add256(P, av.l, 8);
      if (shape & 16u) dot_add256(P, cv.l, 0);
    } else
#pragma unroll 1
    for (uint32_t t = 0; t < nt; t++) {
      const uint4 sl = lds128(tail_s + 16u * (t >> 1));
      const uint32_t lo = (t & 1) ? sl.z : sl.x, ci = (t & 1) ? sl.w : sl.y;
      const uint32_t kind = lo & 0xFu, reg = lo >> 16;
      if (kind == T_MAC) {
        const fe c = const_load(ci);
        const fe x = slot_load(reg);
        dot_mac(P, x.l, c.l);
      } else if (kind == T_CONST) {
        const fe c = const_load(ci);
        dot_add256(P, c.l, 0);
      } else {
        dot_term(P, kind, slot_load(reg), fe_zero());
      }
    }
    R = fe_mont_reduce(P, (int)((ins.y >> 8) & 0xFFu));
  } else if (op == OP_INPUT) {
    R = fe_reduce256(fe_from(__ldg(cx.inputs + 2 * (size_t)ins.y), __ldg(cx.inputs + 2 * (size_t)ins.y + 1)));
  } else if (op == OP_MUL || op == OP_SQR) {
    const fe A = operand(ins.x & F_A_CONST, ins.y);
    R = (op == OP_SQR) ? fe_sqr(A) : fe_mul(A, operand(ins.x & F_B_CONST, ins.z));
  } else if (op == OP_POW5) {
    // Poseidon S-box in one instruction: one fetch, x^2 and x^4 go straight to their witness positions (isa.h)
    const fe A = slot_load(ins.y & 0xFFFFu);
    const uint32_t d4 = ins.y >> 16;
    const fe x2 = fe_sqr(A);
    if (ins.z != NO_POS) { cx.out[2 * (size_t)ins.z] = fe_lo(x2); cx.out[2 * (size_t)ins.z + 1] = fe_hi(x2); }
    const fe x4 = fe_sqr(x2);
    if (d4 != 0xFFFFu) { cx.out[2 * (size_t)(ins.z + d4)] = fe_lo(x4); cx.out[2 * (size_t)(ins.z + d4) + 1] = fe_hi(x4); }
    R = fe_mul(x4, A);
  } else if (op == OP_POW4) {
    // the S-box of a rewritten S-box link (plan.cpp: rewrite_sbox_links): x^2 to the witness, x^4 to its slot and the witness
    const fe x2 = fe_sqr(slot_load(ins.y));
    if (ins.z != NO_POS) { cx.out[2 * (size_t)ins.z] = fe_lo(x2); cx.out[2 * (size_t)ins.z + 1] = fe_hi(x2); }
    R = fe_sqr(x2);
  } else if (op == OP_MULADD) {
    const fe A = operand(ins.x & F_A_CONST, ins.y), Bv = operand(ins.x & F_B_CONST, ins.z), C = operand(ins.x & F_C_CONST, ins.w);
    R = fe_add(fe_mul(A, Bv), C);
  } else if (op == OP_ADD || op == OP_SUB) {
    const fe A = operand(ins.x & F_A_CONST, ins.y), Bv = operand(ins.x & F_B_CONST, ins.z);
    R = (op == OP_ADD) ? fe_add(A, Bv) : fe_sub(A, Bv);
  } else if (op == OP_SHRAND) {
    R = fe_shr_and(slot_load(ins.y), ins.z & 0xFFu, const_load(ins.z >> 8));
  } else {
    fe A = operand(ins.x & F_A_CONST, ins.y), Bv = fe_zero(), C = fe_zero();
    if (op_has_b(op)) Bv = operand(ins.x & F_B_CONST, ins.z);
    if (op == OP_TERN) C = operand(ins.x & F_C_CONST, ins.w);
    fe Rr;                      // its address is taken: keep R itself in registers on the common paths
    lat_exec_rare(op, A, Bv, C, st, &Rr);
    R = Rr;
  }
  if (dst != NO_DST) { sts128(cx.slots_s + 32u * dst, fe_lo(R)); sts128(cx.slots_s + 32u * dst + 16u, fe_hi(R)); }
  if ((ins.x & F_OUT) && op != OP_TERN && op != OP_MULADD && !(cx.dbg & 1u)) { cx.out[2 * (size_t)ins.w] = fe_lo(R); cx.out[2 * (size_t)ins.w + 1] = fe_hi(R); }
}
// one instruction of a slow-warp job: its packet stays in global memory, only the rare operations occur
__device__ __forceinline__ void lat_exec_slow(const LatCtx& cx, const uint4* pk, const uint4 ins, uint32_t* st) {
  const uint32_t op = ins.x & 0xFFu, dst = ins.x >> 16;
  if (op == OP_NOP) return;
  auto operand = [&](uint32_t is_const, uint32_t idx) { return is_const ? fe_from(__ldg(pk + idx), __ldg(pk + idx + 1)) : lds_fe(cx.slots_s + 32u * idx); };
  fe A = operand(ins.x & F_A_CONST, ins.y), Bv = fe_zero(), C = fe_zero(), R;
  if (op_has_b(op)) Bv = operand(ins.x & F_B_CONST, ins.z);
  if (op == OP_TERN) C = operand(ins.x & F_C_CONST, ins.w);
  lat_exec_rare(op, A, Bv, C, st, &R);
  if (dst != NO_DST) { sts128(cx.slots_s + 32u * dst, fe_lo(R)); sts128(cx.slots_s + 32u * dst + 16u, fe_hi(R)); }
  if ((ins.x & F_OUT) && op != OP_TERN) { cx.out[2 * (size_t)ins.w] = fe_lo(R); cx.out[2 * (size_t)ins.w + 1] = fe_hi(R); }
}

// the input set of a latency CTA: 0 for the single-set kernels, row_map[b] or b for CTA b of a batch launch (CTAs of
// different sets share nothing but the read-only plan)
template <bool BATCH, typename P> __device__ __forceinline__ unsigned long long lat_set(const P& p) {
  if (!BATCH) return 0ull;
  return p.row_map ? (unsigned long long)__ldg(p.row_map + blockIdx.x) : (unsigned long long)blockIdx.x;
}

// Dynamic shared memory: [LAT_CTRL_BYTES: control words + mbarriers][n_slots][2] value file | [n_warps][3][LAT_RING_SLOTS] packet rings
template <bool BATCH>
__global__ void __launch_bounds__(LAT_MAX_THREADS) eval_latency_kernel(const LParams p) {
  extern __shared__ uint4 lat_smem[];
  volatile uint32_t* ctrl = reinterpret_cast<volatile uint32_t*>(lat_smem);   // [0] = completed levels, [1 + w] = jobs done by slow warp w
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  const uint32_t smem_s = (uint32_t)__cvta_generic_to_shared(lat_smem);
  const unsigned long long set = lat_set<BATCH>(p);
  uint32_t* const status = (BATCH && p.status) ? p.status + set : p.status;
  if (BATCH && tid == 0 && status) *status = 0;                  // this set's flag word (the single call clears it on the host)
  if (tid < 8) ctrl[tid] = 0;
  if (tid < 3u * p.n_warps) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_s + 32u + 8u * tid) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncthreads();
  uint32_t st = 0;
  LatCtx cx;
  cx.inputs = BATCH ? p.inputs + set * p.I * 2 : p.inputs; cx.out = BATCH ? p.out + set * p.W * 2 : p.out;
  cx.slots_s = smem_s + LAT_CTRL_BYTES; cx.dbg = p.dbg;

  // Packets reach the rings by TMA: ONE bulk copy (cp.async.bulk) per packet, issued by the CONTROL warp (lane w serves
  // main warp w), completing on the mbarrier of the ring stage; the main warps only wait for their barrier, so neither
  // the descriptor walk nor the copy issue is on the path of the warp that holds a level up.
  const uint32_t bar0_s = smem_s + 32u;                          // mbarriers: [main warp][stage], 8 bytes each
  const uint32_t ring0_s = cx.slots_s + 32u * p.n_slots;         // rings: [main warp][stage][LAT_RING_SLOTS]
  auto wait_stage = [&](uint32_t w, uint32_t stage, uint32_t parity) {
    const uint32_t bar = bar0_s + 8u * (3u * w + stage);
    uint32_t done = 0;
    while (!done)
      asm volatile("{ .reg .pred q; mbarrier.try_wait.parity.shared::cta.b64 q, [%1], %2; selp.u32 %0, 1, 0, q; }" : "=r"(done) : "r"(bar), "r"(parity) : "memory");
  };
  if (warp < p.n_warps) {
    const uint32_t nl = p.n_levels;
    const uint32_t bar_threads = (p.n_warps + 1u) * 32u;        // the control warp joins every level barrier
    const uint32_t ring_s = ring0_s + warp * (3u * LAT_RING_SLOTS * 16u);
    uint4 cur = __ldg(p.first + 2 * warp), nxt = __ldg(p.first + 2 * warp + 1);
    uint32_t stage = 0, parity = 0;                  // parity of the stage's current use: flips every third level
    for (uint32_t L = 0; L < nl; L++) {
      wait_stage(warp, stage, parity);                             // this level's packet has landed
      const uint32_t pk_s = ring_s + stage * (LAT_RING_SLOTS * 16u);
      const uint4 desc = lds128(pk_s);                             // {offset, slots, headers, lanes} of the packet two levels ahead
      // header k belongs to lane k mod cur.w; a lane runs its headers in order (a chain: program order, no barrier)
      if (!(p.dbg & 16u) && lane < cur.w) for (uint32_t i = lane; i < cur.z; i += cur.w) lat_exec(cx, pk_s, lds128(pk_s + 16u * (1u + i)), &st);
      __syncwarp();
      lat_level_barrier(bar_threads);
      cur = nxt; nxt = desc;
      if (stage == 2) { stage = 0; parity ^= 1u; } else stage++;
    }
  } else if (warp == p.n_warps) {
    // control warp.  Per level L: (1) lane w reads the descriptor of main warp w's packet L and starts the copy of its
    // packet L + 2 into the stage that level L - 1 used; (2) it waits for the slow-warp jobs whose readers start at
    // level L + 1; (3) it joins the barrier that ends the level and publishes that L + 1 levels are complete.
    const uint32_t nl = p.n_levels, bar_threads = (p.n_warps + 1u) * 32u;
    const bool serve = lane < p.n_warps;
    const uint32_t ring_s = ring0_s + lane * (3u * LAT_RING_SLOTS * 16u);
    auto fetch = [&](const uint4 info, uint32_t stage) {
      const uint32_t bytes = info.y * 16u, bar = bar0_s + 8u * (3u * lane + stage), d = ring_s + stage * (LAT_RING_SLOTS * 16u);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");        // earlier generic reads of the stage vs the async write
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
      if (bytes)
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(d), "l"(p.code + info.x), "r"(bytes), "r"(bar) : "memory");
    };
    if (serve) { fetch(__ldg(p.first + 2 * lane), 0); fetch(__ldg(p.first + 2 * lane + 1), 1); }
    uint32_t stage = 0, parity = 0;
    uint32_t wi = 0;
    uint4 nw = p.n_waits ? __ldg(p.waits) : make_uint4(0xFFFFFFFFu, 0, 0, 0);
    for (uint32_t L = 0; L < nl; L++) {
      if (serve) {
        wait_stage(lane, stage, parity);
        const uint4 desc = lds128(ring_s + stage * (LAT_RING_SLOTS * 16u));
        fetch(desc, stage == 0 ? 2u : stage - 1u);               // stage + 2 mod 3: free since the barrier that ended level L - 1
      }
      __syncwarp();
      while (nw.x == L) {
        flag_wait(smem_s + 4u * (1u + nw.y), nw.z, lane, 40);
        wi++;
        nw = wi < p.n_waits ? __ldg(p.waits + wi) : make_uint4(0xFFFFFFFFu, 0, 0, 0);
      }
      __threadfence_block();
      __syncwarp();                                                // the whole warp arrives at the barrier together
      lat_level_barrier(bar_threads);
      if (lane == 0) { flag_publish(smem_s, L + 1); if (p.level_clock) p.level_clock[L] = clock64(); }
      if (stage == 2) { stage = 0; parity ^= 1u; } else stage++;
    }
  } else if (warp - p.n_warps - 1u < p.n_slow) {
    const uint32_t ws = warp - p.n_warps - 1u;
    const uint32_t nj = __ldg(p.n_jobs + ws);
    const uint4* jq = p.jobs + (size_t)ws * p.max_jobs;
    for (uint32_t j = 0; j < nj; j++) {
      const uint4 job = __ldg(jq + j);                             // {issue level, packet offset, headers, 0}
      const uint4* pk = p.code + job.y;
      const uint4 ins = lane < job.z ? __ldg(pk + 1 + lane) : make_uint4(OP_NOP, 0, 0, 0);
      flag_wait(smem_s, job.x, lane, 100);
      lat_exec_slow(cx, pk, ins, &st);
      __syncwarp();
      if (lane == 0) flag_publish(smem_s + 4u * (1u + ws), j + 1);
    }
  }
  if (status != nullptr && st) atomicOr(status, st);
}

// ---- single-witness latency mode, dataflow plan (plan.hpp: LatencyPlan::dataflow) -----------------------------------
// No level barrier.  Every warp -- the ones that take the long operations included -- walks its own stream of packets:
// chunks of the stream arrive in a 3-stage shared-memory ring by TMA (requested by the warp itself two chunks ahead), a
// packet's wait vector says how many packets of each other warp must be complete before it starts (its operands, and the
// last readers of the values whose slots it overwrites), progress counters in shared memory are published after every
// packet.  Inside a packet one lane = one instruction, as in the level plan; the packets of a warp are ordered by
// __syncwarp.  The plan compiler's emission order makes the waits acyclic (plan.cpp).
struct DParams {
  const uint4* code; const uint32_t* stream_off; const uint32_t* stream_chunks; uint32_t n_warps, chunk_slots;
  const uint4* inputs; uint4* out; uint32_t* status; uint32_t n_slots;
  uint32_t watchdog;       // polls after which a wait gives up (DF_WATCHDOG_SPINS; GW_LAT_WATCHDOG)
  uint32_t dbg;            // GW_LAT_DBG, -DGW_PROFILING experiments: 1 = no witness stores, 2 = publish without fence / atomic, 4 = poll with plain
                           // volatile loads, 8 = fault injection: warp 1's first wait can never be satisfied (watchdog test)
  unsigned long long* clocks; uint32_t clock_rows;   // profiling aid (GW_LAT_CLOCKS, -DGW_PROFILING): [warp][row]{start, after wait, end, first opcode}
  // batch form (BATCH = true): CTA b evaluates input set row_map ? row_map[b] : b; inputs [.][I][2], out [.][W][2], status [.];
  // a CTA whose watchdog fired also sets `aborted` (one word for the launch: the caller's flags are optional)
  const uint32_t* row_map; uint32_t I, W; uint32_t* aborted;
};
static const uint32_t DF_ABORT_WORD = 15;              // control word 15: set by a warp whose wait ran into the watchdog; everybody leaves
static const uint32_t DF_WATCHDOG_SPINS = 1u << 28;    // polls of one wait (tens of seconds: the longest real wait is a Pow, < 1 ms)
static const uint32_t DF_CTRL_BYTES = 384;  // 16 progress words (64 B) + 3 mbarriers x up to 12 warps (288 B), 16 B aligned
// (the "latency plan:" prefix makes gw_calc_witness fall back to the throughput kernel, capi.cpp)
static const char* const LAT_WATCHDOG_ERROR = "latency plan: a packet waited for progress that never came (watchdog); please report the graph";

template <bool BATCH>
__global__ void __launch_bounds__(LAT_MAX_THREADS) eval_dataflow_kernel(const DParams p) {
  extern __shared__ uint4 lat_smem[];
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = __shfl_sync(0xFFFFFFFFu, tid >> 5, 0);   // warp-uniform for the compiler too
  const uint32_t smem_s = (uint32_t)__cvta_generic_to_shared(lat_smem);
  const uint32_t bar0_s = smem_s + 64u;
  const unsigned long long set = lat_set<BATCH>(p);
  uint32_t* const status = (BATCH && p.status) ? p.status + set : p.status;
  if (BATCH && tid == 0 && status) *status = 0;                  // this set's flag word (the single call clears it on the host)
  if (tid < 16) reinterpret_cast<volatile uint32_t*>(lat_smem)[tid] = 0;
  if (tid < 3u * p.n_warps) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0_s + 8u * tid) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncthreads();
  if (warp >= p.n_warps) return;
  uint32_t st = 0;
  LatCtx cx;
  cx.inputs = BATCH ? p.inputs + set * p.I * 2 : p.inputs; cx.out = BATCH ? p.out + set * p.W * 2 : p.out;
  cx.slots_s = smem_s + DF_CTRL_BYTES; cx.dbg = p.dbg;
  const uint32_t chunk_bytes = p.chunk_slots * 16u;
  const uint32_t ring_s = cx.slots_s + 32u * p.n_slots + warp * 3u * chunk_bytes;
  const uint32_t n_chunks = __ldg(p.stream_chunks + warp);
  const uint4* stream = p.code + __ldg(p.stream_off + warp);
  auto request = [&](uint32_t c) {
    if (c >= n_chunks || lane != 0u) return;
    const uint32_t stage = c % 3u, bar = bar0_s + 8u * (3u * warp + stage);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");          // earlier generic reads of the stage vs the async write
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(chunk_bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(ring_s + stage * chunk_bytes), "l"(stream + (size_t)c * p.chunk_slots), "r"(chunk_bytes), "r"(bar) : "memory");
  };
  request(0); request(1);
  for (uint32_t c = 0; c < n_chunks; c++) {
    const uint32_t stage = c % 3u, parity = (c / 3u) & 1u, bar = bar0_s + 8u * (3u * warp + stage);
    uint32_t done = 0;
    while (!done)
      asm volatile("{ .reg .pred q; mbarrier.try_wait.parity.shared::cta.b64 q, [%1], %2; selp.u32 %0, 1, 0, q; }" : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    __syncwarp();                                                         // every lane is done with chunk c - 1: its stage may be refilled
    request(c + 2u);
    uint32_t pk_s = ring_s + stage * chunk_bytes;
    const uint32_t end_s = pk_s + chunk_bytes;
    while (pk_s < end_s) {
      const uint4 desc = lds128(pk_s);            // {slots, headers | lanes << 16, wait vector, packet number}
      if (desc.x == 0u) break;
#ifdef GW_PROFILING
      unsigned long long tc0 = 0, tc1 = 0;
      if (p.clocks) tc0 = clock64();
#endif
      if (desc.z != 0u) {
        // lane k waits for warp k
        if (lane < p.n_warps && lane != warp) {
          uint32_t need;
          asm volatile("ld.shared.u32 %0, [%1];" : "=r"(need) : "r"(pk_s + 16u * desc.z + 4u * lane));
#ifdef GW_PROFILING
          if (need && (p.dbg & 4u)) { uint32_t have; do { asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(have) : "r"(smem_s + 4u * lane) : "memory"); } while (have < need); }
          else
#endif
#ifdef GW_PROFILING
          if ((p.dbg & 8u) && warp == 1u && need) need += 1000000u;
#endif
          if (need) {
            // watchdog: a wait that no packet will ever satisfy (a plan-compiler bug) must end as an error, not as a hung GPU
            uint32_t spins = 0;
            while (flag_read(smem_s + 4u * lane) < need) {
              if ((++spins & 0xFFFFu) == 0u && (flag_read(smem_s + 4u * DF_ABORT_WORD) != 0u || spins > p.watchdog)) {
                flag_publish(smem_s + 4u * DF_ABORT_WORD, 1u);
                break;
              }
            }
          }
        }
        __threadfence_block();                    // acquire: the value-file loads below come after the counters were seen
        __syncwarp();
        if (flag_read(smem_s + 4u * DF_ABORT_WORD) != 0u) {       // warp-uniform: read after the __syncwarp
          if (lane == 0 && status != nullptr) atomicOr(status, 0x80000000u);
          if (BATCH && lane == 0) atomicOr(p.aborted, 1u);
          return;
        }
      }
      const uint32_t nh = desc.y & 0xFFFFu, lanes = desc.y >> 16;
#ifdef GW_PROFILING
      if (p.clocks) tc1 = clock64();
#endif
      if (lane < lanes) for (uint32_t i = lane; i < nh; i += lanes) lat_exec(cx, pk_s, lds128(pk_s + 16u * (1u + i)), &st);
      __syncwarp();
      // release: the value-file stores of all lanes (ordered before lane 0 by __syncwarp) become visible before the counter
#ifdef GW_PROFILING
      if (p.dbg & 2u) { if (lane == 0) asm volatile("st.volatile.shared.u32 [%0], %1;" ::"r"(smem_s + 4u * warp), "r"(desc.w) : "memory"); }
      else
#endif
      if (lane == 0) flag_publish(smem_s + 4u * warp, desc.w);
#ifdef GW_PROFILING
      if (p.clocks && lane == 0 && desc.w <= p.clock_rows) {
        unsigned long long* c = p.clocks + ((size_t)warp * p.clock_rows + (desc.w - 1u)) * 4;
        const uint4 h0 = lds128(pk_s + 16u);
        c[0] = tc0; c[1] = tc1; c[2] = clock64(); c[3] = (unsigned long long)(h0.x & 0xFFu) | ((unsigned long long)lanes << 8) | ((unsigned long long)(h0.y & 0xFFFFFFu) << 16);
      }
#endif
      pk_s += 16u * desc.x;
    }
  }
  if (status != nullptr && st) atomicOr(status, st);
}

// ---- integer-pipe microbenchmark (roofline denominator for multiplication-heavy graphs) ---------
// WHICH = 0: rows of (mad.lo.cc, madc.hi.cc) pairs exactly as in u256_mul_wide -> IMAD.WIDE.U32(.X)
//            with carry predicates; counts one op per 32x32+64 multiply-accumulate,
//         1: mad.lo.u32 (IMAD), 2: mad.hi.u32 (IMAD.HI.U32), 3: add.u32 (ALU pipe, for comparison).
// Every multiplicand comes from another accumulator, so nothing is loop-invariant.  32 ops per
// loop iteration and thread.  Reports executed ops per second over the whole chip.
template <int WHICH>
__global__ void imad_bench_kernel(uint32_t* out, int iters, uint32_t y) {
  uint32_t x = threadIdx.x * 2654435761u + 12345u + blockIdx.x;
  uint32_t s[16];
#pragma unroll
  for (int i = 0; i < 16; i++) s[i] = x + i * 131u;
#pragma unroll 1
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int u = 0; u < 4; u++) {
      if (WHICH == 0) {
#pragma unroll
        for (int r = 0; r < 2; r++) {
          uint32_t* e = s + 8 * r;
          uint32_t m = s[8 * (1 - r) + u];
          asm volatile("mad.lo.cc.u32 %0, %8, %12, %0; madc.hi.cc.u32 %1, %8, %12, %1;"
                       "madc.lo.cc.u32 %2, %9, %12, %2; madc.hi.cc.u32 %3, %9, %12, %3;"
                       "madc.lo.cc.u32 %4, %10, %12, %4; madc.hi.cc.u32 %5, %10, %12, %5;"
                       "madc.lo.cc.u32 %6, %11, %12, %6; madc.hi.u32 %7, %11, %12, %7;"
                       : "+r"(e[0]), "+r"(e[1]), "+r"(e[2]), "+r"(e[3]), "+r"(e[4]), "+r"(e[5]), "+r"(e[6]), "+r"(e[7])
                       : "r"(y), "r"(y ^ 0x55u), "r"(y + 3u), "r"(y * 3u), "r"(m));
        }
      } else {
#pragma unroll
        for (int i = 0; i < 8; i++) {
          if (WHICH == 1) asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+r"(s[i]) : "r"(s[(i + 1) & 7]), "r"(y));
          else if (WHICH == 2) asm volatile("mad.hi.u32 %0, %1, %2, %0;" : "+r"(s[i]) : "r"(s[(i + 1) & 7]), "r"(y));
          else asm volatile("add.u32 %0, %0, %1;" : "+r"(s[i]) : "r"(s[(i + 1) & 7]));
        }
      }
    }
  }
  uint32_t acc = 0;
#pragma unroll
  for (int i = 0; i < 16; i++) acc ^= s[i];
  if (acc == 0x12345678u) out[0] = acc;
}

double imad_microbench(int device, int which) {
  DeviceGuard on(device);
  cudaDeviceProp prop; CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
  uint32_t* d; CUDA_CHECK(cudaMalloc(&d, 4));
  const int iters = 4000, threads = 256, blocks = prop.multiProcessorCount * 8;
  cudaEvent_t e0, e1; CUDA_CHECK(cudaEventCreate(&e0)); CUDA_CHECK(cudaEventCreate(&e1));
  auto go = [&](int n) {
    if (which == 0) imad_bench_kernel<0><<<blocks, threads>>>(d, n, 0x9e3779b9u);
    else if (which == 1) imad_bench_kernel<1><<<blocks, threads>>>(d, n, 0x9e3779b9u);
    else if (which == 2) imad_bench_kernel<2><<<blocks, threads>>>(d, n, 0x9e3779b9u);
    else imad_bench_kernel<3><<<blocks, threads>>>(d, n, 0x9e3779b9u);
  };
  go(50);
  CUDA_CHECK(cudaDeviceSynchronize());
  float best = 1e30f;
  for (int rep = 0; rep < 3; rep++) {
    CUDA_CHECK(cudaEventRecord(e0));
    go(iters);
    CUDA_CHECK(cudaEventRecord(e1));
    CUDA_CHECK(cudaEventSynchronize(e1));
    float ms; CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
    best = std::min(best, ms);
  }
  cudaFree(d); cudaEventDestroy(e0); cudaEventDestroy(e1);
  double ops = (double)blocks * threads * (double)iters * 32.0;
  return ops / (best * 1e-3);
}

// ---- engine ------------------------------------------------------------------------------------------
struct Engine::Dev {
  int device = -1;
  int sms = 0, max_threads = 0;          // threads per CTA the device allows for this plan (one CTA per SM)
  size_t smem_max = 0;
  uint4* code = nullptr; uint4* consts = nullptr;
  uint4* spill = nullptr; size_t spill_threads = 0;
  // every launch of eval_batch_kernel on this device waits for the previous one: they all share the spill area,
  // whatever stream the caller enqueues them on
  cudaEvent_t last_kernel = nullptr;
  // staging for the host-buffer APIs
  cudaStream_t stream[2] = {nullptr, nullptr};
  uint4* d_in[2] = {nullptr, nullptr}; uint4* d_out[2] = {nullptr, nullptr};
  uint32_t* d_status[2] = {nullptr, nullptr};
  uint32_t* d_ff[2] = {nullptr, nullptr};     // lowest violated constraint per set (gw_calc_witness_batch_check only)
  size_t chunk = 0;
  // pinned host ring of the streaming API (three chunks: one in the consumer's hands, one landing, one enqueued)
  uint8_t* h_ring[3] = {nullptr, nullptr, nullptr}; uint32_t* h_flags[3] = {nullptr, nullptr, nullptr};
  size_t h_ring_bytes = 0, h_flags_n = 0;
  // bit-sliced path (bitplan.hpp): program tables, and per-launch scratch that grows with the largest batch seen.
  // bit_fits: the plan's plane file fits this device's shared memory (otherwise every call takes the generic kernels)
  bool bit_fits = false;
  uint4* bit_code = nullptr; uint4* bit_inputs = nullptr; uint32_t* bit_field_inputs = nullptr; uint32_t* bit_field_slots = nullptr; uint32_t bit_n_contract = 0, bit_n_field = 0; int32_t* bit_constpos = nullptr; uint4* bit_consts = nullptr; uint4* bit_wide = nullptr;
  uint32_t* bit_planes = nullptr; uint32_t* bit_ok = nullptr; uint32_t* bit_bad = nullptr; uint32_t* bit_nbad = nullptr;
  size_t bit_groups = 0;
  // feedback for the speculation on the bit contract: how many input sets of the last bit-sliced launch broke it
  uint32_t* bit_nbad_host = nullptr; cudaEvent_t bit_nbad_ev = nullptr; size_t bit_nbad_sets = 0; bool bit_nbad_pending = false;
  // single-witness latency mode
  uint32_t* lat_soff = nullptr; uint32_t* lat_schunks = nullptr;
  uint4* lat_code = nullptr; uint4* lat_first = nullptr; uint4* lat_jobs = nullptr; uint32_t* lat_njobs = nullptr; uint4* lat_waits = nullptr;
  unsigned long long* lat_clock = nullptr;
  uint4* lat_in = nullptr; uint4* lat_out = nullptr; uint32_t* lat_status = nullptr;
  uint32_t* lat_aborted = nullptr;       // latency batch calls: set by a CTA whose watchdog fired (DParams::aborted)
  std::mutex mu;
  ~Dev() {
    int prev = -1;
    cudaGetDevice(&prev);
    cudaSetDevice(device);
    cudaFree(code); cudaFree(consts); cudaFree(spill);
    cudaFree(bit_code); cudaFree(bit_inputs); cudaFree(bit_constpos); cudaFree(bit_consts); cudaFree(bit_wide); cudaFree(bit_field_inputs); cudaFree(bit_field_slots);
    cudaFree(bit_planes); cudaFree(bit_ok); cudaFree(bit_bad); cudaFree(bit_nbad);
    cudaFreeHost(bit_nbad_host); if (bit_nbad_ev) cudaEventDestroy(bit_nbad_ev);
    cudaFree(lat_soff); cudaFree(lat_schunks);
    cudaFree(lat_code); cudaFree(lat_first); cudaFree(lat_jobs); cudaFree(lat_njobs); cudaFree(lat_waits); cudaFree(lat_clock); cudaFree(lat_in); cudaFree(lat_out); cudaFree(lat_status); cudaFree(lat_aborted);
    for (int i = 0; i < 2; i++) { cudaFree(d_in[i]); cudaFree(d_out[i]); cudaFree(d_status[i]); cudaFree(d_ff[i]); if (stream[i]) cudaStreamDestroy(stream[i]); }
    for (int i = 0; i < 3; i++) { cudaFreeHost(h_ring[i]); cudaFreeHost(h_flags[i]); }
    if (last_kernel) cudaEventDestroy(last_kernel);
    if (prev >= 0) cudaSetDevice(prev);
  }
};

static int env_int(const char* name, int dflt) { const char* s = getenv(name); return (s && *s) ? atoi(s) : dflt; }


Engine::Engine(const uint8_t* graph_data, size_t len) {
  graph = deserialize_witnesscalc_graph(graph_data, len);
  init_plan();
}
Engine::Engine(Graph g) : graph(std::move(g)) { init_plan(); }

void Engine::init_plan() {
  max_threads = env_int("GW_THREADS", MAX_THREADS);
  if (max_threads < 32 || max_threads > MAX_THREADS || (max_threads & 31)) throw Error("GW_THREADS must be a multiple of 32 in [32, " + std::to_string(MAX_THREADS) + "]");
  PlanOptions opt; opt.n_regs = (uint32_t)env_int("GW_REGS", (int)opt.n_regs);
  opt.div_batch = (uint32_t)env_int("GW_DIV_BATCH", (int)opt.div_batch);
  opt.fuse_dot = env_int("GW_FUSE_DOT", 1) != 0;
  opt.narrow = env_int("GW_NARROW", 1) != 0;
  opt.fuse_pow5 = env_int("GW_FUSE_POW5", 1) != 0;
  opt.max_terms = (uint32_t)env_int("GW_MAX_TERMS", (int)opt.max_terms);
  plan = compile_plan(graph, opt);
  // Boolean graphs get a bit-sliced plan as well (exact for every input: input sets that are not bits fall back to `plan`)
  if (env_int("GW_BITSLICE", 1) != 0) {
    BitPlanOptions bo;
    bo.max_slots = (uint32_t)env_int("GW_BIT_MAX_SLOTS", (int)bo.max_slots);
    bo.merge_luts = env_int("GW_BIT_MERGE", 1) != 0;
    bit_plan = compile_bit_plan(graph, bo);
  }
}

// shared memory of a CTA of T threads without the hot-constant area: instruction rings + register file
static size_t smem_base(const Plan& plan, int T) { return (size_t)(T / 32) * RING * 16 + (size_t)plan.n_regs * 32 * T; }
// shared memory of one warp's plane file in bit_eval_kernel (the ring variants add mbarriers and header chunks behind it)
static size_t bit_plane_bytes(const BitPlan& bp) { return ((size_t)bp.n_slots * 4 + 15) & ~(size_t)15; }

// Launch geometry for a batch of B input sets: one persistent CTA per SM; T = the smallest multiple of 32 that
// covers the batch in the fewest waves of full CTAs.
int Engine::threads_for(size_t B, int sms, int t_max) const {
  const size_t per_wave = (size_t)sms * t_max;
  const size_t waves = (B + per_wave - 1) / per_wave;
  size_t t = (B + (size_t)sms * waves - 1) / ((size_t)sms * waves);
  t = (t + 31) / 32 * 32;
  return (int)std::min<size_t>(std::max<size_t>(t, 32), (size_t)t_max);
}

Engine::~Engine() = default;

Engine::Dev* Engine::dev(int device) {
  std::lock_guard<std::mutex> lk(mu);
  auto it = devs.find(device);
  if (it != devs.end()) return it->second.get();
  check_device(device);
  DeviceGuard on(device);
  std::unique_ptr<Dev> d(new Dev());
  d->device = device;
  cudaDeviceProp prop; CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
  d->sms = prop.multiProcessorCount;
  d->smem_max = prop.sharedMemPerBlockOptin;
  cudaFuncAttributes fa; CUDA_CHECK(cudaFuncGetAttributes(&fa, eval_batch_kernel));
  int t_max = std::min(max_threads, (int)(prop.regsPerBlock / std::max(fa.numRegs, 1)) / 32 * 32);
  while (t_max >= 32 && smem_base(plan, t_max) > d->smem_max) t_max -= 32;
  if (t_max < 32) throw Error("register file does not fit shared memory: lower GW_REGS");
  d->max_threads = t_max;
  CUDA_CHECK(cudaFuncSetAttribute(eval_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)d->smem_max));
  CUDA_CHECK(cudaFuncSetAttribute(eval_dataflow_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)d->smem_max));
  CUDA_CHECK(cudaFuncSetAttribute(eval_latency_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)d->smem_max));   // per device, not per graph
  // batch forms: as many CTAs per SM as shared memory holds (two of a small graph), so the carveout goes to shared memory
  CUDA_CHECK(cudaFuncSetAttribute(eval_dataflow_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)d->smem_max));
  CUDA_CHECK(cudaFuncSetAttribute(eval_latency_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)d->smem_max));
  CUDA_CHECK(cudaFuncSetAttribute(eval_dataflow_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
  CUDA_CHECK(cudaFuncSetAttribute(eval_latency_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
  CUDA_CHECK(cudaEventCreateWithFlags(&d->last_kernel, cudaEventDisableTiming));
  CUDA_CHECK(cudaMalloc(&d->code, plan.code.size() * sizeof(Instr)));
  CUDA_CHECK(cudaMemcpy(d->code, plan.code.data(), plan.code.size() * sizeof(Instr), cudaMemcpyHostToDevice));
  CUDA_CHECK(cudaMalloc(&d->consts, plan.consts.size() * 32));
  CUDA_CHECK(cudaMemcpy(d->consts, plan.consts.data(), plan.consts.size() * 32, cudaMemcpyHostToDevice));
  d->spill_threads = (size_t)d->sms * t_max;
  if (plan.n_spill || plan.n_spill_narrow) CUDA_CHECK(cudaMalloc(&d->spill, ((size_t)plan.n_spill * 32 + (size_t)plan.n_spill_narrow * 8) * d->spill_threads));
  d->bit_fits = use_bit_path() && bit_plane_bytes(bit_plan) <= d->smem_max;
  if (d->bit_fits) {
    const BitPlan& bp = bit_plan;
    CUDA_CHECK(cudaFuncSetAttribute(bit_eval_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)d->smem_max));
    CUDA_CHECK(cudaFuncSetAttribute(bit_eval_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)d->smem_max));
    CUDA_CHECK(cudaFuncSetAttribute(bit_eval_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)d->smem_max));
    CUDA_CHECK(cudaMalloc(&d->bit_code, bp.code.size() * sizeof(BitOp)));
    CUDA_CHECK(cudaMemcpy(d->bit_code, bp.code.data(), bp.code.size() * sizeof(BitOp), cudaMemcpyHostToDevice));
    // input list as 16-byte entries, the contract inputs first (the batch kernel reads those and takes the field inputs
    // from the per-bit slot tables; the single-set kernel walks the whole list)
    std::vector<uint32_t> quads, finputs, fslots;
    for (int pass = 0; pass < 2; pass++)
      for (size_t k = 0; k + 2 < bp.inputs.size(); k += 3) {
        const bool contract = bp.inputs[k + 2] == BIT_CONTRACT;
        if (contract != (pass == 0)) continue;
        quads.push_back(bp.inputs[k]); quads.push_back(bp.inputs[k + 1]); quads.push_back(bp.inputs[k + 2]); quads.push_back(0);
        if (contract) { d->bit_n_contract++; continue; }
        if (finputs.empty() || finputs.back() != bp.inputs[k]) { finputs.push_back(bp.inputs[k]); fslots.resize(fslots.size() + 256, BIT_NO_SLOT); }
        if (bp.inputs[k + 2] < 256) fslots[(finputs.size() - 1) * 256 + bp.inputs[k + 2]] = bp.inputs[k + 1];
      }
    d->bit_n_field = (uint32_t)finputs.size();
    CUDA_CHECK(cudaMalloc(&d->bit_field_inputs, std::max<size_t>(finputs.size(), 1) * 4));
    CUDA_CHECK(cudaMemcpy(d->bit_field_inputs, finputs.data(), finputs.size() * 4, cudaMemcpyHostToDevice));
    CUDA_CHECK(cudaMalloc(&d->bit_field_slots, std::max<size_t>(fslots.size(), 1) * 4));
    CUDA_CHECK(cudaMemcpy(d->bit_field_slots, fslots.data(), fslots.size() * 4, cudaMemcpyHostToDevice));
    CUDA_CHECK(cudaMalloc(&d->bit_inputs, std::max<size_t>(quads.size(), 4) * 4));
    CUDA_CHECK(cudaMemcpy(d->bit_inputs, quads.data(), quads.size() * 4, cudaMemcpyHostToDevice));
    quads.clear();
    for (size_t k = 0; k + 2 < bp.wide.size(); k += 3) { quads.push_back(bp.wide[k]); quads.push_back(bp.wide[k + 1]); quads.push_back(bp.wide[k + 2]); quads.push_back(0); }
    CUDA_CHECK(cudaMalloc(&d->bit_wide, std::max<size_t>(quads.size(), 4) * 4));
    CUDA_CHECK(cudaMemcpy(d->bit_wide, quads.data(), quads.size() * 4, cudaMemcpyHostToDevice));
    CUDA_CHECK(cudaMalloc(&d->bit_constpos, std::max<size_t>(bp.const_of_pos.size(), 1) * 4));
    CUDA_CHECK(cudaMemcpy(d->bit_constpos, bp.const_of_pos.data(), bp.const_of_pos.size() * 4, cudaMemcpyHostToDevice));
    CUDA_CHECK(cudaMalloc(&d->bit_consts, std::max<size_t>(bp.const_vals.size(), 1) * 32));
    CUDA_CHECK(cudaMemcpy(d->bit_consts, bp.const_vals.data(), bp.const_vals.size() * 32, cudaMemcpyHostToDevice));
    CUDA_CHECK(cudaMalloc(&d->bit_nbad, 4));
    CUDA_CHECK(cudaHostAlloc(&d->bit_nbad_host, 4, cudaHostAllocDefault));
    CUDA_CHECK(cudaEventCreateWithFlags(&d->bit_nbad_ev, cudaEventDisableTiming));
  }
  return (devs[device] = std::move(d)).get();
}

// Enqueues one eval_batch_kernel on `stream`, behind every earlier launch of this engine on the device (the spill
// area is indexed by resident thread and shared by all launches).  Callers hold d->mu.
// Bit-sliced path: pack + contract check + LUT steps (bit_eval_kernel), expansion of the plane words to witness rows
// (bit_expand_kernel), then the generic kernel for the input sets that are not bits (usually none: an empty launch).
void Engine::launch_bit(Dev* d, const void* d_inputs, size_t B, void* d_witness, uint32_t* d_status, void* stream) {
  const BitPlan& bp = bit_plan;
  cudaStream_t s = (cudaStream_t)stream;
  const size_t n_groups = (B + 31) / 32;
  if (n_groups > 0x7FFFFFFFull) throw Error("batch too large");
  CUDA_CHECK(cudaStreamWaitEvent(s, d->last_kernel, 0));
  if (n_groups > d->bit_groups) {
    // scratch of the largest batch seen; cudaFree waits for the kernels that still use the old one
    cudaFree(d->bit_planes); d->bit_planes = nullptr; cudaFree(d->bit_ok); d->bit_ok = nullptr; cudaFree(d->bit_bad); d->bit_bad = nullptr;
    d->bit_groups = 0;
    CUDA_CHECK(cudaMalloc(&d->bit_planes, n_groups * (size_t)std::max<uint32_t>(bp.plane_stride, 1) * 4));
    CUDA_CHECK(cudaMalloc(&d->bit_ok, n_groups * 4));
    CUDA_CHECK(cudaMalloc(&d->bit_bad, n_groups * 32 * 4));
    d->bit_groups = n_groups;
  }
  // the count of an earlier launch may still be on its way to the host (launch() copies it after recording last_kernel,
  // on that launch's stream): it has to land before this launch zeroes and recounts it
  CUDA_CHECK(cudaStreamWaitEvent(s, d->bit_nbad_ev, 0));
  CUDA_CHECK(cudaMemsetAsync(d->bit_nbad, 0, 4, s));
  BParams q;
  q.code = d->bit_code; q.n_steps = bp.n_steps; q.n_slots = bp.n_slots;
  q.in_list = d->bit_inputs; q.n_in = (uint32_t)(bp.inputs.size() / 3); q.n_contract = d->bit_n_contract;
  q.field_inputs = d->bit_field_inputs; q.n_field = d->bit_n_field; q.field_slots = d->bit_field_slots;
  q.inputs = (const uint4*)d_inputs; q.I = bp.n_inputs; q.W = bp.n_witness; q.B = B; q.n_groups = (uint32_t)n_groups;
  q.planes = d->bit_planes; q.plane_stride = bp.plane_stride; q.ok_words = d->bit_ok; q.bad_list = d->bit_bad; q.n_bad = d->bit_nbad; q.status = d_status;
  // shared memory per warp (group): the plane file, and for the ring variants 3 mbarriers + 3 chunks of LUT headers
  const size_t planes_b = bit_plane_bytes(bp);
  const size_t single_b = planes_b + 32 + 3 * (size_t)BIT_CHUNK_SINGLE * 512, ring_b = planes_b + 32 + 3 * (size_t)BIT_CHUNK_BATCH * 512;
  if (planes_b > d->smem_max) throw Error("bit-sliced plan: plane file does not fit shared memory");     // callers check d->bit_fits
  // GW_TRACE_HOST=1: which variant of bit_eval_kernel ran, in what shape
  const bool trace = env_int("GW_TRACE_HOST", 0) != 0;
  if (B == 1 && single_b <= d->smem_max) {
    q.warp_bytes = (uint32_t)single_b;
    bit_eval_kernel<true, true><<<1, 32, single_b, s>>>(q);
    if (trace) fprintf(stderr, "[gw bit] variant single, warps 1, ctas 1, groups 1\n");
  } else {
    // ring variant unless it would leave an SM with fewer resident groups than the batch can give it (GW_BIT_RING=0/1 forces)
    const int env_ring = env_int("GW_BIT_RING", -1);
    const size_t fit_ring = d->smem_max / ring_b, fit_reg = d->smem_max / planes_b;
    const size_t per_sm = (n_groups + (size_t)d->sms - 1) / (size_t)d->sms;
    // (a short program -- Num2Bits: 24 steps -- is over before a ring pays for its set-up: measured, profiles/r02k)
    bool ring = ring_b <= d->smem_max && bp.n_steps >= 128 && (per_sm <= fit_ring || fit_ring * 2 >= fit_reg);
    if (env_ring == 0) ring = false; else if (env_ring == 1 && ring_b <= d->smem_max) ring = true;
    const size_t wb = ring ? ring_b : planes_b;
    // warps per CTA: as many as shared memory allows, but enough CTAs to cover the SMs twice
    int wpb = (int)std::min<size_t>(8, d->smem_max / wb);
    while (wpb > 1 && n_groups < (size_t)wpb * 2 * (size_t)d->sms) wpb--;
    const int env_wpb = env_int("GW_BIT_WARPS", 0);
    if (env_wpb >= 1 && env_wpb <= wpb) wpb = env_wpb;
    q.warp_bytes = (uint32_t)wb;
    const unsigned grid = (unsigned)((n_groups + wpb - 1) / wpb);
    if (ring) bit_eval_kernel<false, true><<<grid, wpb * 32, (size_t)wpb * wb, s>>>(q);
    else bit_eval_kernel<false, false><<<grid, wpb * 32, (size_t)wpb * wb, s>>>(q);
    if (trace) fprintf(stderr, "[gw bit] variant %s, warps %d, ctas %u, groups %zu\n", ring ? "ring" : "reg", wpb, grid, n_groups);
  }
  CUDA_CHECK(cudaGetLastError());
  const uint32_t tiles = (bp.n_witness + 31) / 32;
  const unsigned long long n_warp_tiles = (unsigned long long)n_groups * tiles;
  if (n_warp_tiles) {
    bit_expand_kernel<<<(unsigned)((n_warp_tiles + 7) / 8), 256, 0, s>>>(d->bit_planes, d->bit_ok, d->bit_constpos, d->bit_consts, (uint4*)d_witness,
                                                                        bp.n_witness, bp.plane_stride, (uint32_t)n_groups, tiles);
    CUDA_CHECK(cudaGetLastError());
  }
  const uint32_t n_wide = (uint32_t)(bp.wide.size() / 3);
  if (n_wide) {
    const unsigned long long n_warps = (unsigned long long)n_groups * n_wide;
    bit_expand_wide_kernel<<<(unsigned)((n_warps + 7) / 8), 256, 0, s>>>(d->bit_planes, d->bit_ok, d->bit_wide, n_wide, (uint32_t*)d_witness,
                                                                        bp.n_witness, bp.plane_stride, (uint32_t)n_groups);
    CUDA_CHECK(cudaGetLastError());
  }
}

void Engine::launch(Dev* d, const void* d_inputs, size_t B, void* d_witness, uint32_t* d_status, void* stream) {
  if (B == 0) return;
  if (plan.code.empty()) {            // an empty witness (gw_graph_select of no position): nothing to run, no set is flagged
    if (d_status) CUDA_CHECK(cudaMemsetAsync(d_status, 0, B * 4, (cudaStream_t)stream));
    return;
  }
  // The bit-sliced plan speculates that the inputs under its contract are bits.  When most input sets of a launch were
  // not (somebody feeds field elements to a graph that would also work on bits), the speculation is dropped for this
  // graph: such batches would pay for both paths.  The count arrives asynchronously; it is looked at on the next launch.
  if (d->bit_nbad_pending && cudaEventQuery(d->bit_nbad_ev) == cudaSuccess) {
    d->bit_nbad_pending = false;
    if (d->bit_nbad_sets >= 64 && (size_t)*d->bit_nbad_host * 2 > d->bit_nbad_sets) bit_disabled.store(true);
  }
  const bool bit = d->bit_fits && !bit_disabled.load() && B >= (size_t)env_int("GW_BIT_MIN_SETS", 1);
  if (bit) launch_bit(d, d_inputs, B, d_witness, d_status, stream);
  KParams p;
  p.row_map = bit ? d->bit_bad : nullptr; p.n_dev = bit ? d->bit_nbad : nullptr;
  p.code = d->code; p.n_slots = (uint32_t)plan.code.size(); p.consts = d->consts;
  p.inputs = (const uint4*)d_inputs; p.out = (uint4*)d_witness; p.spill = d->spill; p.status = d_status;
  p.nspill = reinterpret_cast<uint2*>(d->spill + (size_t)plan.n_spill * 2 * d->spill_threads);
  p.B = B; p.I = plan.n_inputs; p.W = plan.n_witness;
  const int T = threads_for(B, d->sms, d->max_threads);
  size_t n_tiles = (B + T - 1) / T;
  if (n_tiles > 0xFFFFFFFFull) throw Error("batch too large");
  p.n_tiles = (uint32_t)n_tiles;
  p.spill_threads = d->spill_threads;
#ifdef GW_PROFILING
  p.out_wrap = (unsigned long long)env_int("GW_DEBUG_OUT_WRAP", 0);
#endif
  // whatever shared memory the rings and the register file leave goes to the most used constants
  const size_t base = smem_base(plan, T);
  p.n_hot = (uint32_t)std::min<size_t>(plan.consts.size(), (d->smem_max - base) / 32);
  if (env_int("GW_HOT_CONSTS", -1) >= 0) p.n_hot = std::min<uint32_t>(p.n_hot, (uint32_t)env_int("GW_HOT_CONSTS", 0));
  const int grid = (int)std::min<size_t>(n_tiles, (size_t)d->sms);
  CUDA_CHECK(cudaStreamWaitEvent((cudaStream_t)stream, d->last_kernel, 0));
  eval_batch_kernel<<<grid, T, base + (size_t)p.n_hot * 32, (cudaStream_t)stream>>>(p);
  CUDA_CHECK(cudaGetLastError());
  CUDA_CHECK(cudaEventRecord(d->last_kernel, (cudaStream_t)stream));
  if (bit && !d->bit_nbad_pending) {
    CUDA_CHECK(cudaMemcpyAsync(d->bit_nbad_host, d->bit_nbad, 4, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CUDA_CHECK(cudaEventRecord(d->bit_nbad_ev, (cudaStream_t)stream));
    d->bit_nbad_sets = B; d->bit_nbad_pending = true;
  }
}

int Engine::device_max_threads(int device) { return dev(device)->max_threads; }

void Engine::run_device(int device, const void* d_inputs, size_t B, void* d_witness, uint32_t* d_status, void* stream) {
  Dev* d = dev(device);
  DeviceGuard on(device);
  std::lock_guard<std::mutex> lk(d->mu);     // enqueue order = execution order of the kernels (launch() chains them)
  launch(d, d_inputs, B, d_witness, d_status, stream);
}

// device staging buffers of the host-buffer APIs, two of each, for chunks of `chunk` input sets
void Engine::ensure_staging(Dev* d, size_t chunk) {
  if (chunk <= d->chunk) return;
  const size_t in_b = (size_t)plan.n_inputs * 32, out_b = (size_t)plan.n_witness * 32;
  // the old buffers go first (they can be most of HBM); the bookkeeping is cleared before anything can throw
  d->chunk = 0;
  for (int i = 0; i < 2; i++) {
    cudaFree(d->d_in[i]); d->d_in[i] = nullptr;
    cudaFree(d->d_out[i]); d->d_out[i] = nullptr;
    cudaFree(d->d_status[i]); d->d_status[i] = nullptr;
    cudaFree(d->d_ff[i]); d->d_ff[i] = nullptr;
  }
  for (int i = 0; i < 2; i++) {
    CUDA_CHECK(cudaMalloc(&d->d_in[i], std::max<size_t>(chunk * in_b, 32)));
    CUDA_CHECK(cudaMalloc(&d->d_out[i], std::max<size_t>(chunk * out_b, 32)));
    CUDA_CHECK(cudaMalloc(&d->d_status[i], chunk * 4));
    if (!d->stream[i]) CUDA_CHECK(cudaStreamCreateWithFlags(&d->stream[i], cudaStreamNonBlocking));
  }
  d->chunk = chunk;
}

namespace {
// GW_TRACE_HOST=1: device-side timeline of a host-buffer call (per chunk: start, inputs landed, kernel done, witness landed)
struct HostTrace {
  bool on; std::vector<cudaEvent_t> ev;
  HostTrace() : on(env_int("GW_TRACE_HOST", 0) != 0) {}
  void mark(cudaStream_t st) { if (on) { cudaEvent_t e; if (cudaEventCreate(&e) == cudaSuccess) { cudaEventRecord(e, st); ev.push_back(e); } } }
  void print(int device, size_t B, size_t chunk) {
    if (!on) return;
    fprintf(stderr, "[gw trace] device %d: %zu sets, chunk %zu:", device, B, chunk);
    for (size_t i = 0; i < ev.size(); i++) { float ms = 0; cudaEventElapsedTime(&ms, ev[0], ev[i]); fprintf(stderr, "%s%.1f", i % 4 == 0 ? " | " : " ", ms); }
    fprintf(stderr, " ms\n");
  }
  ~HostTrace() { for (cudaEvent_t e : ev) cudaEventDestroy(e); }
};
}  // namespace

// host buffers: chunked, double-buffered H2D -> kernel -> D2H on two streams (latency: the latency kernels, one CTA per set)
void Engine::run_host_on(int device, const uint8_t* inputs, size_t B, uint8_t* witness, uint32_t* status, size_t out_pitch,
                         R1cs* check, uint32_t* first_failed, bool latency) {
  Dev* d = dev(device);
  DeviceGuard on(device);
  std::lock_guard<std::mutex> lk(d->mu);
  const size_t in_b = (size_t)plan.n_inputs * 32, out_b = (size_t)plan.n_witness * 32;
  if (out_pitch == 0) out_pitch = out_b;
  if (out_pitch < out_b) throw Error("witness pitch is smaller than a witness row");
  // chunk size: bounded by a device-memory budget per staging buffer (two of them), at most two full
  // waves of resident threads, and small enough to give the copy/compute pipeline >= 4 stages when the
  // batch is large.  GW_CHUNK_MB overrides the budget.
  size_t free_b = 0, total_b = 0;
  CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
  size_t budget = (size_t)env_int("GW_CHUNK_MB", 24576) << 20;
  budget = std::min(budget, (free_b + 2 * d->chunk * (in_b + out_b)) / 5);
  size_t chunk = budget / std::max<size_t>(out_b + in_b, 1);
  if (latency) {
    // latency kernels: whole waves of resident CTAs (what the budget holds if that is less than one wave)
    const size_t wave = latency_wave(d);
    if (chunk >= wave) chunk = chunk / wave * wave;
    if (B >= 4 * wave) chunk = std::min(chunk, ((B + 3) / 4 + wave - 1) / wave * wave);
  } else {
    chunk = std::min<size_t>(chunk, 2 * d->spill_threads);
    if (B >= 4 * 2048) chunk = std::min(chunk, (B + 3) / 4);
  }
  chunk = std::max<size_t>(std::min(chunk, B), 1);
  ensure_staging(d, chunk);
  if (check)                                   // verdict buffers of the staging chunk size, allocated on the first check
    for (int i = 0; i < 2; i++) if (!d->d_ff[i]) CUDA_CHECK(cudaMalloc(&d->d_ff[i], d->chunk * 4));
  // The kernels of consecutive chunks run back to back (launch() chains them: one spill area) while the copies
  // of the two streams overlap with them.
  HostTrace tr;
  StreamDrain drain{d->stream[0], d->stream[1]};
  if (latency) { latency_arm(d, d->stream[0]); CUDA_CHECK(cudaStreamSynchronize(d->stream[0])); }
  int k = 0;
  for (size_t off = 0; off < B; off += chunk, k ^= 1) {
    size_t nb = std::min(chunk, B - off);
    cudaStream_t s = d->stream[k];
    tr.mark(s);
    CUDA_CHECK(cudaMemcpyAsync(d->d_in[k], inputs + off * in_b, nb * in_b, cudaMemcpyHostToDevice, s));
    tr.mark(s);
    if (latency) latency_launch(d, d->d_in[k], nb, d->d_out[k], status ? d->d_status[k] : nullptr, s);
    else launch(d, d->d_in[k], nb, d->d_out[k], status ? d->d_status[k] : nullptr, s);
    if (check) {
      // the chunk's witness rows are checked where they are; only the verdicts have to cross PCIe
      check->check_device(device, d->d_out[k], nb, out_b, d->d_ff[k], s);
      CUDA_CHECK(cudaMemcpyAsync(first_failed + off, d->d_ff[k], nb * 4, cudaMemcpyDeviceToHost, s));
    }
    tr.mark(s);
    if (!witness) {}      // gw_calc_witness_batch_check without witness: the rows stay on the device
    else if (out_pitch == out_b) CUDA_CHECK(cudaMemcpyAsync(witness + off * out_b, d->d_out[k], nb * out_b, cudaMemcpyDeviceToHost, s));
    else if (out_b) CUDA_CHECK(cudaMemcpy2DAsync(witness + off * out_pitch, out_pitch, d->d_out[k], out_b, out_b, nb, cudaMemcpyDeviceToHost, s));
    if (status) CUDA_CHECK(cudaMemcpyAsync(status + off, d->d_status[k], nb * 4, cudaMemcpyDeviceToHost, s));
    tr.mark(s);
  }
  CUDA_CHECK(cudaStreamSynchronize(d->stream[0]));
  CUDA_CHECK(cudaStreamSynchronize(d->stream[1]));
  if (latency) latency_check(d);
  tr.print(device, B, chunk);
}

void Engine::run_host(const uint8_t* inputs, size_t B, uint8_t* witness, uint32_t* status, int n_gpus, int first_device, size_t out_pitch,
                      R1cs* check, uint32_t* first_failed, bool latency) {
  if (B == 0) return;
  if (out_pitch == 0) out_pitch = (size_t)plan.n_witness * 32;
  if (n_gpus <= 1) { run_host_on(first_device, inputs, B, witness, status, out_pitch, check, first_failed, latency); return; }
  const size_t in_b = (size_t)plan.n_inputs * 32;
  run_shards(B, n_gpus, first_device, [&](int device, size_t lo, size_t hi) {
    run_host_on(device, inputs + lo * in_b, hi - lo, witness ? witness + lo * out_pitch : nullptr, status ? status + lo : nullptr,
                out_pitch, check, check ? first_failed + lo : nullptr, latency);
  });
}

// Streaming output path: the witnesses of the batch never exist in host memory all at once.  Per GPU, chunk k's rows
// go kernel -> device staging buffer (k mod 2) -> pinned ring slot (k mod 3); the consumer sees chunk k - 1 while
// chunk k lands and chunk k + 1 is enqueued, so the device-to-host engine never waits for the host.
void Engine::stream_on(int device, const uint8_t* inputs, size_t B, size_t first_set, size_t chunk_req, const ChunkFn& fn) {
  Dev* d = dev(device);
  DeviceGuard on(device);
  std::lock_guard<std::mutex> lk(d->mu);
  const size_t in_b = (size_t)plan.n_inputs * 32, out_b = std::max<size_t>((size_t)plan.n_witness * 32, 32);
  // chunk: a ring slot of GW_STREAM_CHUNK_MB (default 8 GiB; three slots are pinned per GPU), a device staging budget
  // like run_host_on's, at most one full wave of resident threads; whole warps
  size_t free_b = 0, total_b = 0;
  CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
  const size_t dev_budget = (free_b + 2 * d->chunk * (in_b + out_b)) / 5;
  size_t chunk = chunk_req;
  if (chunk == 0) {
    const size_t slot = (size_t)env_int("GW_STREAM_CHUNK_MB", 8192) << 20;
    chunk = std::min<size_t>(std::min(slot, dev_budget) / out_b, d->spill_threads);
    if (chunk >= 64) chunk = chunk / 32 * 32;
  }
  chunk = std::max<size_t>(std::min(std::min(chunk, dev_budget / (in_b + out_b)), B), 1);
  ensure_staging(d, chunk);
  if (chunk * out_b > d->h_ring_bytes || chunk > d->h_flags_n) {
    d->h_ring_bytes = 0; d->h_flags_n = 0;
    for (int i = 0; i < 3; i++) { cudaFreeHost(d->h_ring[i]); d->h_ring[i] = nullptr; cudaFreeHost(d->h_flags[i]); d->h_flags[i] = nullptr; }
    for (int i = 0; i < 3; i++) {
      CUDA_CHECK(cudaHostAlloc(&d->h_ring[i], chunk * out_b, cudaHostAllocDefault));
      CUDA_CHECK(cudaHostAlloc(&d->h_flags[i], chunk * 4, cudaHostAllocDefault));
    }
    d->h_ring_bytes = chunk * out_b; d->h_flags_n = chunk;
  }
  struct Events {
    cudaEvent_t e[3] = {nullptr, nullptr, nullptr};
    ~Events() { for (cudaEvent_t x : e) if (x) cudaEventDestroy(x); }
  } landed;
  for (int i = 0; i < 3; i++) CUDA_CHECK(cudaEventCreateWithFlags(&landed.e[i], cudaEventDisableTiming));
  HostTrace tr;
  StreamDrain drain{d->stream[0], d->stream[1]};
  auto deliver = [&](size_t k) {
    const size_t off = k * chunk, nb = std::min(chunk, B - off);
    CUDA_CHECK(cudaEventSynchronize(landed.e[k % 3]));
    if (fn(device, first_set + off, nb, d->h_ring[k % 3], (size_t)plan.n_witness * 32, d->h_flags[k % 3]) != 0) throw Error("witness stream stopped by the consumer");
  };
  size_t k = 0;
  for (size_t off = 0; off < B; off += chunk, k++) {
    const size_t nb = std::min(chunk, B - off);
    const int sb = (int)(k & 1), slot = (int)(k % 3);
    cudaStream_t s = d->stream[sb];
    tr.mark(s);
    CUDA_CHECK(cudaMemcpyAsync(d->d_in[sb], inputs + off * in_b, nb * in_b, cudaMemcpyHostToDevice, s));
    tr.mark(s);
    launch(d, d->d_in[sb], nb, d->d_out[sb], d->d_status[sb], s);
    tr.mark(s);
    if (plan.n_witness) CUDA_CHECK(cudaMemcpyAsync(d->h_ring[slot], d->d_out[sb], nb * (size_t)plan.n_witness * 32, cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaMemcpyAsync(d->h_flags[slot], d->d_status[sb], nb * 4, cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaEventRecord(landed.e[slot], s));
    tr.mark(s);
    if (k >= 1) deliver(k - 1);
  }
  if (k >= 1) deliver(k - 1);
  tr.print(device, B, chunk);
}

void Engine::run_stream(const uint8_t* inputs, size_t B, int n_gpus, int first_device, size_t chunk_sets, const ChunkFn& fn) {
  if (B == 0) return;
  if (n_gpus < 1) n_gpus = 1;
  // always on worker threads: they are pinned near their GPU before the ring is allocated, the caller's affinity is left alone
  const size_t in_b = (size_t)plan.n_inputs * 32;
  run_shards(B, n_gpus, first_device, [&](int device, size_t lo, size_t hi) { stream_on(device, inputs + lo * in_b, hi - lo, lo, chunk_sets, fn); });
}

// shared memory of one latency CTA of plan lp (engine.cu: eval_dataflow_kernel, eval_latency_kernel)
static size_t latency_smem(const LatencyPlan& lp) {
  if (lp.dataflow) return DF_CTRL_BYTES + (size_t)lp.n_slots * 32 + (size_t)lp.n_phys_warps * 3 * lp.chunk_slots * 16;
  return ((size_t)lp.n_slots * 2 + LAT_CTRL_BYTES / 16 + (size_t)lp.n_warps * 3 * LAT_RING_SLOTS) * 16;
}
static int latency_threads(const LatencyPlan& lp) { return (int)(lp.dataflow ? lp.n_phys_warps : lp.n_warps + 1 + lp.n_slow_warps) * 32; }

// The latency plan of the graph and its tables on d's device, for the single call and the batch alike: compiled once, under
// the GW_LAT_* options of that moment (a compile error -- "graph is too wide" -- is remembered and given to every later
// call), uploaded once per device.  Callers hold d->mu.
const LatencyPlan& Engine::latency_plan(Dev* d) {
  {
    std::lock_guard<std::mutex> lk2(mu);
    if (!lat_error.empty()) throw Error(lat_error);
    if (!lat_ready) {
      LatencyOptions lo;
      // GW_LAT_MODE=level: the level-synchronous plan (control warp, CTA barrier per level); default: the dataflow plan
      const char* lat_mode = getenv("GW_LAT_MODE");
      lo.dataflow = !(lat_mode && strcmp(lat_mode, "level") == 0);
      // dataflow: no control warp
      // (measured on authV2, profiles/r02o: 6 + 3 warps 16.3 ms, 7 + 3: 16.9, 8 + 4: 17.6, 7 + 3 with warp 0 alone on its
      // sub-partition: 18.1 -- every extra warp of dependent carry chains slows its sub-partition's other warps down)
      lo.n_warps = (uint32_t)env_int("GW_LAT_WARPS", lo.dataflow ? 6 : (int)lo.n_warps);
      lo.n_slow_warps = (uint32_t)env_int("GW_LAT_SLOW_WARPS", lo.dataflow ? 3 : (int)lo.n_slow_warps);
      lo.exclusive_warp0 = env_int("GW_LAT_EXCL", 0) != 0;
      lo.packet_slots = LAT_RING_SLOTS;
      const size_t df_rings = std::min<size_t>(12, lo.n_warps + lo.n_slow_warps + (lo.exclusive_warp0 ? 2 : 0));     // physical warps, empty ones included
      if (lo.dataflow) lo.max_slots = (uint32_t)std::min<size_t>((d->smem_max / 16 - DF_CTRL_BYTES / 16 - df_rings * 3 * LAT_RING_SLOTS) / 2, 0xFFFF);
      else
      lo.max_slots = (uint32_t)std::min<size_t>((d->smem_max / 16 - LAT_CTRL_BYTES / 16 - (size_t)lo.n_warps * 3 * LAT_RING_SLOTS) / 2, 0xFFFF);
      lo.slow_levels = (uint32_t)env_int("GW_LAT_D", 0);
      lo.split_dot = env_int("GW_LAT_SPLIT", 1) != 0;
      lo.fuse = env_int("GW_LAT_FUSE", 1) != 0;
      lo.sbox_links = env_int("GW_LAT_LINKS", 1) != 0;           // 0: never, 1: where the timing model prefers it, 2: always
      lo.force_sbox_links = env_int("GW_LAT_LINKS", 1) == 2;
      lo.chain = env_int("GW_LAT_CHAIN", 1) != 0;
      if (!lo.dataflow && (lo.n_warps + 1 + lo.n_slow_warps) * 32 > (uint32_t)LAT_MAX_THREADS) throw Error("GW_LAT_WARPS + GW_LAT_SLOW_WARPS must not exceed 11");
      try { lat_plan = compile_latency_plan(graph, lo); }
      catch (const Error& e) { lat_error = e.what(); throw; }
      lat_ready = true;
    }
  }
  const LatencyPlan& lp = lat_plan;
  if (!d->lat_code) {
    CUDA_CHECK(cudaMalloc(&d->lat_code, std::max<size_t>(lp.code.size(), 1) * sizeof(Instr)));
    CUDA_CHECK(cudaMemcpy(d->lat_code, lp.code.data(), lp.code.size() * sizeof(Instr), cudaMemcpyHostToDevice));
    if (lp.dataflow) {
      const uint32_t NW = lp.n_phys_warps;
      CUDA_CHECK(cudaMalloc(&d->lat_soff, NW * 4)); CUDA_CHECK(cudaMalloc(&d->lat_schunks, NW * 4));
      CUDA_CHECK(cudaMemcpy(d->lat_soff, lp.stream_off.data(), NW * 4, cudaMemcpyHostToDevice));
      CUDA_CHECK(cudaMemcpy(d->lat_schunks, lp.stream_chunks.data(), NW * 4, cudaMemcpyHostToDevice));
    } else {
      CUDA_CHECK(cudaMalloc(&d->lat_first, std::max<size_t>(lp.first.size(), 4) * 4));
      CUDA_CHECK(cudaMemcpy(d->lat_first, lp.first.data(), lp.first.size() * 4, cudaMemcpyHostToDevice));
      CUDA_CHECK(cudaMalloc(&d->lat_jobs, std::max<size_t>(lp.jobs.size(), 4) * 4));
      CUDA_CHECK(cudaMemcpy(d->lat_jobs, lp.jobs.data(), lp.jobs.size() * 4, cudaMemcpyHostToDevice));
      CUDA_CHECK(cudaMalloc(&d->lat_njobs, std::max<size_t>(lp.n_jobs.size(), 1) * 4));
      CUDA_CHECK(cudaMemcpy(d->lat_njobs, lp.n_jobs.data(), lp.n_jobs.size() * 4, cudaMemcpyHostToDevice));
      CUDA_CHECK(cudaMalloc(&d->lat_waits, std::max<size_t>(lp.waits.size(), 4) * 4));
      CUDA_CHECK(cudaMemcpy(d->lat_waits, lp.waits.data(), lp.waits.size() * 4, cudaMemcpyHostToDevice));
#ifdef GW_PROFILING
      if (env_int("GW_LAT_CLOCKS", 0) != 0) CUDA_CHECK(cudaMalloc(&d->lat_clock, ((size_t)lp.n_levels + 1) * 8));
#endif
    }
  }
  return lp;
}

// one witness, host buffers: inputs I x 32 B, witness W x 32 B; returns the kernel time in ms if asked
void Engine::run_latency(int device, const uint8_t* inputs, uint8_t* witness, uint32_t* status, float* kernel_ms) {
  Dev* d = dev(device);
  if (plan.code.empty()) {            // an empty witness: no kernel, no set flagged
    if (status) *status = 0;
    if (kernel_ms) *kernel_ms = 0;
    return;
  }
  DeviceGuard on(device);
  std::lock_guard<std::mutex> lk(d->mu);
  if (!d->lat_in) {
    CUDA_CHECK(cudaMalloc(&d->lat_in, std::max<size_t>((size_t)plan.n_inputs * 32, 32)));
    CUDA_CHECK(cudaMalloc(&d->lat_out, std::max<size_t>((size_t)plan.n_witness * 32, 32)));
    CUDA_CHECK(cudaMalloc(&d->lat_status, 4));
  }
  // Boolean graphs: the bit-sliced plan IS the level-parallel plan -- its steps are up to 32 independent LUT nodes, one
  // node per lane, values in a shared-memory plane file, __syncwarp between steps (no CTA barrier, no packets).  One
  // input set occupies bit 0 of every plane word.  SHA-256(512): 8 058 steps against 7 010 levels of 256-bit
  // instructions in the generic latency plan.  An input set that breaks the bit contract takes the generic plan below.
  if (d->bit_fits && bit_path_active() && bit_plan.n_luts > 0 && env_int("GW_LAT_BIT", 1) != 0) {     // pure wiring (Num2Bits alone): three launches cost more than the generic kernel
    CUDA_CHECK(cudaMemcpyAsync(d->lat_in, inputs, (size_t)plan.n_inputs * 32, cudaMemcpyHostToDevice, 0));
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (kernel_ms) { CUDA_CHECK(cudaEventCreate(&e0)); CUDA_CHECK(cudaEventCreate(&e1)); CUDA_CHECK(cudaEventRecord(e0, 0)); }
    launch_bit(d, d->lat_in, 1, d->lat_out, d->lat_status, nullptr);
    CUDA_CHECK(cudaEventRecord(d->last_kernel, 0));
    if (kernel_ms) CUDA_CHECK(cudaEventRecord(e1, 0));
    uint32_t n_bad = 0;
    CUDA_CHECK(cudaMemcpy(&n_bad, d->bit_nbad, 4, cudaMemcpyDeviceToHost));     // 4 bytes decide which buffer is worth copying
    if (kernel_ms) { CUDA_CHECK(cudaEventElapsedTime(kernel_ms, e0, e1)); cudaEventDestroy(e0); cudaEventDestroy(e1); }
    if (n_bad == 0) {
      CUDA_CHECK(cudaMemcpy(witness, d->lat_out, (size_t)plan.n_witness * 32, cudaMemcpyDeviceToHost));
      if (status) *status = 0;
      return;
    }
  }
  const LatencyPlan& lp = latency_plan(d);
  const size_t in_b = (size_t)lp.n_inputs * 32;
  if (lp.dataflow) {
    const uint32_t NW = lp.n_phys_warps;
    DParams q;
    q.code = d->lat_code; q.stream_off = d->lat_soff; q.stream_chunks = d->lat_schunks; q.n_warps = NW; q.chunk_slots = lp.chunk_slots;
    q.inputs = d->lat_in; q.out = d->lat_out; q.status = d->lat_status; q.n_slots = lp.n_slots;
    q.row_map = nullptr; q.I = q.W = 0; q.aborted = nullptr;
    const size_t smem_df = latency_smem(lp);
    q.clocks = nullptr; q.clock_rows = 0; q.dbg = 0;
    q.watchdog = (uint32_t)env_int("GW_LAT_WATCHDOG", (int)DF_WATCHDOG_SPINS);
#ifdef GW_PROFILING
    q.dbg = (uint32_t)env_int("GW_LAT_DBG", 0);
#endif
#ifdef GW_PROFILING
    unsigned long long* d_clk = nullptr;
    uint32_t max_rows = 0;
    if (env_int("GW_LAT_CLOCKS", 0) != 0) {
      // rows per warp are not stored in the plan: bound them by the packets in the streams
      max_rows = (uint32_t)std::min<uint64_t>(lp.n_rows, 1u << 20);
      CUDA_CHECK(cudaMalloc(&d_clk, (size_t)NW * max_rows * 32));
      CUDA_CHECK(cudaMemset(d_clk, 0, (size_t)NW * max_rows * 32));
      q.clocks = d_clk; q.clock_rows = max_rows;
    }
#endif
    CUDA_CHECK(cudaMemcpyAsync(d->lat_in, inputs, in_b, cudaMemcpyHostToDevice, 0));
    CUDA_CHECK(cudaMemsetAsync(d->lat_status, 0, 4, 0));
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (kernel_ms) { CUDA_CHECK(cudaEventCreate(&e0)); CUDA_CHECK(cudaEventCreate(&e1)); CUDA_CHECK(cudaEventRecord(e0, 0)); }
    eval_dataflow_kernel<false><<<1, NW * 32, smem_df, 0>>>(q);
    CUDA_CHECK(cudaGetLastError());
    if (kernel_ms) CUDA_CHECK(cudaEventRecord(e1, 0));
    uint32_t h_status = 0;
    CUDA_CHECK(cudaMemcpyAsync(witness, d->lat_out, (size_t)lp.n_witness * 32, cudaMemcpyDeviceToHost, 0));
    CUDA_CHECK(cudaMemcpyAsync(&h_status, d->lat_status, 4, cudaMemcpyDeviceToHost, 0));
    CUDA_CHECK(cudaStreamSynchronize(0));
    if (kernel_ms) { CUDA_CHECK(cudaEventElapsedTime(kernel_ms, e0, e1)); cudaEventDestroy(e0); cudaEventDestroy(e1); }
    // (the "latency plan:" prefix makes gw_calc_witness fall back to the throughput kernel, capi.cpp)
    if (h_status & 0x80000000u) throw Error(LAT_WATCHDOG_ERROR);
    if (status) *status = h_status;
#ifdef GW_PROFILING
    if (d_clk) {
      // GW_LAT_CLOCKS=1: one line per packet "warp row start wait_end end opcode lanes" (cycles since the first packet)
      std::vector<unsigned long long> c((size_t)NW * max_rows * 4);
      CUDA_CHECK(cudaMemcpy(c.data(), d_clk, c.size() * 8, cudaMemcpyDeviceToHost));
      cudaFree(d_clk);
      const char* path = getenv("GW_LAT_CLOCKS_FILE");
      FILE* f = fopen(path && *path ? path : "gw_lat_clocks.txt", "w");
      if (f) {
        unsigned long long t0 = ~0ull;
        for (size_t k = 0; k < c.size(); k += 4) if (c[k + 2] && c[k] < t0) t0 = c[k];
        for (uint32_t w = 0; w < NW; w++)
          for (uint32_t r = 0; r < max_rows; r++) {
            const unsigned long long* e = &c[((size_t)w * max_rows + r) * 4];
            if (!e[2]) break;
            fprintf(f, "%u %u %llu %llu %llu %llu %llu %llx\n", w, r, e[0] - t0, e[1] - t0, e[2] - t0, e[3] & 0xFF, (e[3] >> 8) & 0xFF, e[3] >> 16);
          }
        fclose(f);
      }
    }
#endif
    return;
  }
  const size_t smem = latency_smem(lp);
#ifdef GW_PROFILING
  const bool clocks = env_int("GW_LAT_CLOCKS", 0) != 0;
#else
  const bool clocks = false;
#endif
  if (lp.n_levels == 0) return;
  LParams p;
  p.code = d->lat_code; p.first = d->lat_first; p.n_levels = lp.n_levels; p.n_warps = lp.n_warps; p.n_slots = lp.n_slots;
  p.jobs = d->lat_jobs; p.n_jobs = d->lat_njobs; p.max_jobs = lp.max_jobs; p.n_slow = lp.n_slow_warps;
  p.waits = d->lat_waits; p.n_waits = (uint32_t)(lp.waits.size() / 4);
  p.inputs = d->lat_in; p.out = d->lat_out; p.status = status ? d->lat_status : nullptr;
  p.level_clock = d->lat_clock;
  p.row_map = nullptr; p.I = p.W = 0;
  p.dbg = 0;
#ifdef GW_PROFILING
  p.dbg = (uint32_t)env_int("GW_LAT_DBG", 0);      // timing experiments: -DGW_PROFILING builds only
#endif
  CUDA_CHECK(cudaMemcpyAsync(d->lat_in, inputs, in_b, cudaMemcpyHostToDevice, 0));
  if (status) CUDA_CHECK(cudaMemsetAsync(d->lat_status, 0, 4, 0));
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (kernel_ms) { CUDA_CHECK(cudaEventCreate(&e0)); CUDA_CHECK(cudaEventCreate(&e1)); CUDA_CHECK(cudaEventRecord(e0, 0)); }
  eval_latency_kernel<false><<<1, (lp.n_warps + 1 + lp.n_slow_warps) * 32, smem, 0>>>(p);
  CUDA_CHECK(cudaGetLastError());
  if (kernel_ms) CUDA_CHECK(cudaEventRecord(e1, 0));
  CUDA_CHECK(cudaMemcpyAsync(witness, d->lat_out, (size_t)lp.n_witness * 32, cudaMemcpyDeviceToHost, 0));
  if (status) CUDA_CHECK(cudaMemcpyAsync(status, d->lat_status, 4, cudaMemcpyDeviceToHost, 0));
  CUDA_CHECK(cudaStreamSynchronize(0));
  if (kernel_ms) { CUDA_CHECK(cudaEventElapsedTime(kernel_ms, e0, e1)); cudaEventDestroy(e0); cudaEventDestroy(e1); }
  if (clocks && d->lat_clock) {
    // GW_LAT_CLOCKS=1: cycles per level to stderr-readable file gw_lat_clocks.txt (tools/gpu_latency.py reads it)
    std::vector<unsigned long long> c((size_t)lp.n_levels);
    CUDA_CHECK(cudaMemcpy(c.data(), d->lat_clock, c.size() * 8, cudaMemcpyDeviceToHost));
    const char* path = getenv("GW_LAT_CLOCKS_FILE");
    FILE* f = fopen(path && *path ? path : "gw_lat_clocks.txt", "w");
    if (f) {            // cycles per level
      for (size_t k = 1; k < lp.n_levels; k++) fprintf(f, "%llu\n", c[k] - c[k - 1]);
      fclose(f);
    }
  }
}

// Boolean graphs take the bit-sliced plan in latency mode, as the single call decides (Engine::run_latency)
bool Engine::latency_bit(Dev* d) const { return d->bit_fits && bit_path_active() && bit_plan.n_luts > 0 && env_int("GW_LAT_BIT", 1) != 0; }

// input sets one wave of latency_launch holds on d's device: one CTA per set, as many per SM as registers and shared
// memory allow (the bit-sliced plan: 32 sets per warp, a warp per SM and wave at least)
size_t Engine::latency_wave(Dev* d) {
  if (latency_bit(d)) return (size_t)d->sms * 32;
  const LatencyPlan& lp = latency_plan(d);
  int per_sm = 0;
  if (lp.dataflow) CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, eval_dataflow_kernel<true>, latency_threads(lp), latency_smem(lp)));
  else CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, eval_latency_kernel<true>, latency_threads(lp), latency_smem(lp)));
  return (size_t)d->sms * (size_t)std::max(per_sm, 1);
}

// n input sets, one latency CTA each: CTA b evaluates set row_map ? row_map[b] : b of d_inputs / d_witness / d_status.
// Chained behind every earlier launch of this engine on the device, as launch() is.  Callers hold d->mu.
void Engine::latency_kernels(Dev* d, const void* d_inputs, size_t n, const uint32_t* row_map, void* d_witness, uint32_t* d_status, void* stream) {
  const LatencyPlan& lp = latency_plan(d);
  cudaStream_t s = (cudaStream_t)stream;
  if (n > 0x7FFFFFFFull) throw Error("batch too large");
  CUDA_CHECK(cudaStreamWaitEvent(s, d->last_kernel, 0));
  if (lp.dataflow) {
    DParams q;
    q.code = d->lat_code; q.stream_off = d->lat_soff; q.stream_chunks = d->lat_schunks; q.n_warps = lp.n_phys_warps; q.chunk_slots = lp.chunk_slots;
    q.inputs = (const uint4*)d_inputs; q.out = (uint4*)d_witness; q.status = d_status; q.n_slots = lp.n_slots;
    q.watchdog = (uint32_t)env_int("GW_LAT_WATCHDOG", (int)DF_WATCHDOG_SPINS);
    q.dbg = 0; q.clocks = nullptr; q.clock_rows = 0;
    q.row_map = row_map; q.I = lp.n_inputs; q.W = lp.n_witness; q.aborted = d->lat_aborted;
    eval_dataflow_kernel<true><<<(unsigned)n, latency_threads(lp), latency_smem(lp), s>>>(q);
  } else {
    LParams p;
    p.code = d->lat_code; p.first = d->lat_first; p.n_levels = lp.n_levels; p.n_warps = lp.n_warps; p.n_slots = lp.n_slots;
    p.jobs = d->lat_jobs; p.n_jobs = d->lat_njobs; p.max_jobs = lp.max_jobs; p.n_slow = lp.n_slow_warps;
    p.waits = d->lat_waits; p.n_waits = (uint32_t)(lp.waits.size() / 4);
    p.inputs = (const uint4*)d_inputs; p.out = (uint4*)d_witness; p.status = d_status;
    p.level_clock = nullptr; p.dbg = 0;
    p.row_map = row_map; p.I = lp.n_inputs; p.W = lp.n_witness;
    eval_latency_kernel<true><<<(unsigned)n, latency_threads(lp), latency_smem(lp), s>>>(p);
  }
  CUDA_CHECK(cudaGetLastError());
  CUDA_CHECK(cudaEventRecord(d->last_kernel, s));
}

// gw_calc_witness_latency for n input sets on `stream` (d_status optional): what the single call does for one set, for
// every set of the batch.  A Boolean graph runs all n sets bit-sliced, then the sets that broke the bit contract through
// the latency kernels (a 4-byte readback decides).  Callers hold d->mu; the watchdog is checked by latency_check.
void Engine::latency_launch(Dev* d, const void* d_inputs, size_t n, void* d_witness, uint32_t* d_status, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (n == 0) return;
  if (plan.code.empty()) {            // an empty witness: no kernel, no set flagged
    if (d_status) CUDA_CHECK(cudaMemsetAsync(d_status, 0, n * 4, s));
    return;
  }
  if (latency_bit(d)) {
    launch_bit(d, d_inputs, n, d_witness, d_status, s);
    CUDA_CHECK(cudaEventRecord(d->last_kernel, s));
    uint32_t n_bad = 0;
    CUDA_CHECK(cudaMemcpyAsync(&n_bad, d->bit_nbad, 4, cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
    if (n_bad != 0) latency_kernels(d, d_inputs, n_bad, d->bit_bad, d_witness, d_status, s);
    return;
  }
  latency_kernels(d, d_inputs, n, nullptr, d_witness, d_status, s);
}

// clears the watchdog word of d's device before a latency batch call (ordered before its kernels on `s`)
void Engine::latency_arm(Dev* d, void* stream) {
  if (!d->lat_aborted) CUDA_CHECK(cudaMalloc(&d->lat_aborted, 4));
  CUDA_CHECK(cudaMemsetAsync(d->lat_aborted, 0, 4, (cudaStream_t)stream));
}
// after the call's work is complete: fails the call when a CTA's watchdog fired
void Engine::latency_check(Dev* d) {
  uint32_t aborted = 0;
  CUDA_CHECK(cudaMemcpy(&aborted, d->lat_aborted, 4, cudaMemcpyDeviceToHost));
  if (aborted) throw Error(LAT_WATCHDOG_ERROR);
}

void Engine::run_latency_device(int device, const void* d_inputs, size_t n, void* d_witness, uint32_t* d_status, void* stream) {
  if (n == 0) return;
  Dev* d = dev(device);
  DeviceGuard on(device);
  std::lock_guard<std::mutex> lk(d->mu);
  cudaStream_t s = (cudaStream_t)stream;
  latency_arm(d, s);
  latency_launch(d, d_inputs, n, d_witness, d_status, s);
  CUDA_CHECK(cudaStreamSynchronize(s));
  latency_check(d);
}

}  // namespace gw
