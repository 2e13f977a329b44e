// A circuit's rank-1 constraint system (iden3 .r1cs, version 1), compiled once into a device program that checks
// witness rows: for every constraint k, <A_k,w> * <B_k,w> - <C_k,w> == 0 (mod M).  The wire numbering of the R1CS is
// the witness numbering of the graph (circom writes both), so wire i is witness position i.
//
// Program (r1cs_eval.cuh executes it): a stream of 8-byte items (two uint32).  Per constraint a 16-byte header
// {n_a, n_b}, {n_c, 0}, then the n_a + n_b + n_c terms of A, B and C.  A term is {wire, meta}:
//   meta = kind[1:0] | n_cond_sub[3:2] | constant index << 4
// kind is an isa.h TermKind (T_MAC, T_ADDHI, T_SUBHI).  n_cond_sub != 0 marks the last term of a chunk: the 512-bit
// accumulator is Montgomery-reduced there (fe_mont_reduce with that many conditional subtractions) and added to the
// linear combination's partial sum.  The constant table holds c * 2^256 mod M (the OP_DOT convention), most used first.
#pragma once
#include <stdint.h>

#include <map>
#include <memory>
#include <mutex>
#include <vector>

#include "graph.hpp"

namespace gw {

static const uint32_t R1CS_OK = 0xFFFFFFFFu;        // GW_R1CS_OK: every constraint holds
static const uint32_t R1CS_ABC_GROTH16 = 1u;        // GW_R1CS_ABC_GROTH16: the ABC vectors in the Groth16 domain layout

struct R1csHeader {
  uint32_t n8 = 0, n_wires = 0, n_pub_out = 0, n_pub_in = 0, n_prv_in = 0, n_constraints = 0;
  uint64_t n_labels = 0;
};

struct R1csProgram {
  std::vector<uint32_t> code;       // item k = code[2k], code[2k + 1]
  std::vector<U256> consts;         // pre-scaled, most used first
  uint64_t n_terms = 0, n_mac_terms = 0, n_chunks = 0;
};

// Term weights of the chunk bound, in thousandths of M (see r1cs.cpp: lc_chunk_bound).
static const uint32_t R1CS_W_BASE = 1000, R1CS_W_MAC = 190, R1CS_W_HI = 1000, R1CS_W_MAX = 5250;
// conditional subtractions that bring a chunk of total weight w (<= R1CS_W_MAX) to [0, M)
static inline uint32_t r1cs_cond_subs(uint32_t w) { return w <= 2000 ? 1u : w <= 4000 ? 2u : 3u; }

// parses an .r1cs file and compiles its constraints; throws gw::Error on a malformed file
void parse_r1cs(const uint8_t* data, size_t len, R1csHeader& hdr, R1csProgram& prog);

class R1cs {
 public:
  R1cs(const uint8_t* data, size_t len);
  ~R1cs();
  R1cs(const R1cs&) = delete;

  R1csHeader hdr;
  R1csProgram prog;

  // rows resident on `device`: row r at d_witness + r * row_pitch (row_pitch >= n_wires * 32, a multiple of 16);
  // d_first_failed[r] = lowest violated constraint or R1CS_OK.  Asynchronous on `stream`.
  void check_device(int device, const void* d_witness, size_t B, size_t row_pitch, uint32_t* d_first_failed, void* stream);
  // host rows (row r at witness + r * row_pitch), sharded over n_gpus devices starting at first_device
  void check_host(const uint8_t* witness, size_t B, size_t row_pitch, uint32_t* first_failed, int n_gpus, int first_device);

  // <A_k,w>, <B_k,w>, <C_k,w> per row (gw_r1cs_abc_batch): row r of the output at abc + r * abc_pitch is A | B | C, each
  // abc_len(options) entries of 32 bytes.  first_failed (optional) receives the check's verdicts.
  // entries per vector: n_constraints, or with R1CS_ABC_GROTH16 the smallest power of two >= n_constraints + n_pub + 1
  uint64_t abc_len(uint32_t options) const;
  // checks the layout arguments (device: 16-byte multiples too) without touching a device; returns 3 x n x 32
  size_t abc_row_bytes(size_t row_pitch, size_t abc_pitch, uint32_t options, bool device) const;
  void abc_device(int device, const void* d_witness, size_t B, size_t row_pitch, void* d_abc, size_t abc_pitch, uint32_t options,
                  uint32_t* d_first_failed, void* stream);
  void abc_host(const uint8_t* witness, size_t B, size_t row_pitch, uint8_t* abc, size_t abc_pitch, uint32_t options,
                uint32_t* first_failed, int n_gpus, int first_device);

  // Groth16 quotient evaluations per row (gw_r1cs_quotient_batch): with n = abc_len(R1CS_ABC_GROTH16) and X_odd the
  // coset forward transform of the inverse transform of X (ntt.hpp), h_i = A_odd[i] * B_odd[i] - C_odd[i].
  // Device: abc_device into the work rows (d_work + r * work_pitch, work_pitch >= 3 x n x 32), then the transforms in
  // place, all on `stream`; h is left in the first n x 32 bytes of each work row.  Host: h row r at h + r * h_pitch.
  // checks the layout arguments without touching a device; returns log2(n)
  uint32_t quotient_log_n(size_t row_pitch, size_t out_pitch, bool device) const;
  void quotient_device(int device, const void* d_witness, size_t B, size_t row_pitch, void* d_work, size_t work_pitch,
                       uint32_t* d_first_failed, void* stream);
  void quotient_host(const uint8_t* witness, size_t B, size_t row_pitch, uint8_t* h, size_t h_pitch, uint32_t* first_failed,
                     int n_gpus, int first_device);

 private:
  struct Dev;
  struct Launch;
  struct AbcOut { uint8_t* abc; size_t pitch; uint32_t options; bool quotient; };   // quotient: h only (n x 32 bytes per row)
  Dev* dev(int device);
  Launch launch(Dev* d, const void* d_witness, size_t B, size_t row_pitch, uint32_t* d_first_failed) const;
  void host_rows_on(int device, const uint8_t* witness, size_t B, size_t row_pitch, uint32_t* first_failed, const AbcOut* out);
  void host_rows(const uint8_t* witness, size_t B, size_t row_pitch, uint32_t* first_failed, const AbcOut* out, int n_gpus,
                 int first_device);
  std::map<int, std::unique_ptr<Dev>> devs;
  std::mutex mu;
};

}  // namespace gw
