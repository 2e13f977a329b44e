/* C ABI of the B200 witness evaluator.
 *
 * Part 1 is the reference's header verbatim in meaning: /root/reference/include/graph_witness.h:7-28
 * (GW_ERROR_CODE, gw_status_t, gw_calc_witness, gw_free_status), implemented by the reference in
 * src/lib.rs:28-111.  tests/csrc/reference_abi_part1.c checks it against the reference's declarations.
 * Part 2 is the batch extension (SURVEY.md section 8b): load a graph once, evaluate many input sets.
 *
 * Every entry point is backed by CUDA kernels; there is no CPU fallback: without a usable GPU the
 * calls return 1 with an error message.
 */
#include <stddef.h>
#include <stdint.h>
#include <stdlib.h>

#ifndef RUST_GRAPH_WITNESS_H
#define RUST_GRAPH_WITNESS_H

#ifdef __cplusplus
extern "C" {
#endif

/* ---- part 1: drop-in (reference include/graph_witness.h:7-28) ---------------------------------- */

typedef enum {
  OK = 0,
  ERROR = 1
} GW_ERROR_CODE;

typedef struct {
  GW_ERROR_CODE code;
  char *error_msg;
} gw_status_t;

/* inputs: NUL-terminated UTF-8 JSON; graph_data: a wtns.graph.001 file; on success *wtns_data is a
 * malloc'ed .wtns file of *wtns_len bytes that the caller frees.  Returns 0 on success, 1 on error
 * (status->code = ERROR, status->error_msg malloc'ed).  Deviation from src/lib.rs:106-108: on
 * success status is {OK, NULL} (the reference writes {ERROR, "test error"}) and nothing is printed. */
int
gw_calc_witness(const char *inputs,
                const void *graph_data, const size_t graph_data_len,
                void **wtns_data, size_t *wtns_len,
                const gw_status_t *status);

/* reference include/graph_witness.h:23-28 defines this function in the header; kept, but static
 * inline so that the header can be included from more than one translation unit. */
static inline void
gw_free_status(gw_status_t *status) {
  if (status->error_msg != NULL) {
    free(status->error_msg);
  }
}

/* ---- part 2: batch extension ---------------------------------------------------------------------- */

typedef struct gw_graph gw_graph_t;

typedef struct {
  uint64_t n_nodes;       /* nodes in the graph file */
  uint64_t n_ops;         /* Op + UnoOp + TresOp nodes (unit of the node-ops/s metric) */
  uint32_t n_inputs;      /* I: input buffer length including slot 0 (the constant 1) */
  uint32_t n_witness;     /* W: witness length */
  uint32_t n_input_signals;
  uint32_t n_instrs;      /* device instructions per witness */
  uint32_t n_regs;        /* per-witness registers in shared memory */
  uint32_t n_spill;       /* per-witness spill slots in HBM */
  uint64_t n_mul;         /* live Mul nodes of the graph (field multiplications per witness, algorithmic) */
  uint64_t n_div;         /* live Div nodes of the graph (field divisions per witness, algorithmic) */
  uint64_t n_spill_ld;    /* spill loads per witness */
  uint64_t n_spill_st;    /* spill stores per witness */
  /* what the plan compiler made of it (per witness) */
  uint32_t n_slots;       /* 16-byte program slots */
  uint32_t n_dot;         /* fused linear combinations (one Montgomery reduction each) */
  uint32_t n_dot_mac;     /* value x constant products inside them */
  uint32_t n_mul_instr;   /* value x value multiplications (Barrett) */
  uint32_t n_inversions;  /* modular inversions after Div batching */
  uint32_t threads;       /* threads per CTA */
  uint32_t sets_per_thread; /* input sets evaluated per thread */
  uint32_t n_narrow_instr; /* instructions computed on int64 (values the plan compiler proves to be small, isa.h F_NARROW) */
  /* bit-sliced plan (Boolean graphs: 32 input sets per machine word, one 3-input LUT per lane) */
  uint32_t bit_eligible;  /* 1: batch launches of this graph run bit-sliced (input sets that break the bit contract: generic kernel) */
  uint32_t bit_luts;      /* LUT instructions per group of 32 input sets */
  uint32_t bit_steps;     /* steps of 32 LUTs */
  uint32_t bit_wide;      /* witness values assembled from several planes (Bits2Num sums, field inputs passed through) */
} gw_graph_info_t;

/* replaces storage::deserialize_witnesscalc_graph (src/storage.rs:214-249) + upload; parse once */
int gw_graph_load(const void *graph_data, size_t graph_data_len, gw_graph_t **graph, gw_status_t *status);
void gw_graph_free(gw_graph_t *graph);
int gw_graph_info(const gw_graph_t *graph, gw_graph_info_t *info);
/* i-th input signal of the graph's input map (InputSignalsInfo, src/lib.rs:19); name is owned by the graph */
int gw_graph_input_signal(const gw_graph_t *graph, uint32_t i, const char **name, uint32_t *offset, uint32_t *len);

/* calc_witness (src/lib.rs:125-136) + wtns_from_witness (:114-123) on a pre-loaded graph */
int gw_graph_calc_witness(gw_graph_t *graph, const char *inputs_json, void **wtns_data, size_t *wtns_len,
                          gw_status_t *status);

/* graph::evaluate (src/graph.rs:367-391) for n_sets independent input sets, HOST buffers.
 *   inputs : n_sets x n_inputs x 32 bytes, little-endian 256-bit values, row-major; slot 0 of every
 *            row is ignored (it is the constant 1); values >= M are reduced mod M like Fr::new.
 *   witness: n_sets x n_witness x 32 bytes, canonical little-endian (the .wtns payload of each set).
 *   flags  : optional (may be NULL) n_sets x uint32: per-set bits for cases where the reference
 *            panics (1 Shl overflow, 2 Bor/Bxor == M, 4 Pow, 8 Id, 16 Lnot/Bnot).
 *   n_gpus : the sets are split into n_gpus contiguous shards, one per device, no collective. */
int gw_calc_witness_batch(gw_graph_t *graph, const uint8_t *inputs, size_t n_sets, uint8_t *witness,
                          uint32_t *flags, int n_gpus, gw_status_t *status);

/* same on devices first_device .. first_device + n_gpus - 1: for hosts that run one process per GPU (each process
 * passes its own device) or that keep some devices for other work. */
int gw_calc_witness_batch_on(gw_graph_t *graph, int first_device, const uint8_t *inputs, size_t n_sets,
                             uint8_t *witness, uint32_t *flags, int n_gpus, gw_status_t *status);

/* same, buffers already resident on CUDA device `device`; enqueued on `cuda_stream` (a cudaStream_t,
 * NULL = default stream) and asynchronous with respect to the host. */
int gw_calc_witness_batch_device(gw_graph_t *graph, int device, const void *d_inputs, size_t n_sets,
                                 void *d_witness, uint32_t *d_flags, void *cuda_stream, gw_status_t *status);

/* Calls on one graph and device may come from any thread and any stream: the library runs the kernels of one graph
 * on one device one after the other (they share a per-device scratch area), in the order the calls were made. */

/* single-witness latency mode (BASELINE config 5): ONE input set (n_inputs x 32 B, host), parallel across the nodes
 * of the graph's dependency levels; witness is n_witness x 32 B (host).  *kernel_ms (optional) receives the device time
 * of the kernels alone.
 *   - Boolean graphs (SHA-256, Num2Bits, comparators; gw_graph_info_t.bit_luts > 0) run their bit-sliced plan with
 *     one warp: a step = up to 32 independent LUT nodes, one per lane.  An input set that breaks the plan's contract
 *     (an input that must be 0 or 1 and is not) is evaluated by the generic kernel below in the same call.
 *   - everything else: one CTA; every warp walks its own stream of packets (one instruction per lane), packets wait on
 *     progress counters of the other warps; the long operations (Div, Pow, Idiv, Mod) have warps of their own.
 * Fails with "latency plan: graph is too wide ..." when the values alive at once do not fit the shared memory of one
 * SM.  gw_calc_witness / gw_graph_calc_witness use this mode for their single witness and fall back to the throughput
 * kernel with a batch of one in that case. */
int gw_calc_witness_latency(gw_graph_t *graph, int device, const uint8_t *inputs, uint8_t *witness, uint32_t *flags,
                            float *kernel_ms, gw_status_t *status);

/* gw_calc_witness_latency for n_sets input sets: one latency-mode CTA per set, as many at once as the device holds.
 * Row r of witness / flags is byte-identical to gw_calc_witness_latency on input row r.  Host buffers as
 * gw_calc_witness_batch (inputs n_sets x n_inputs x 32 B, witness n_sets x n_witness x 32 B, flags optional),
 * sharded over devices first_device .. first_device + n_gpus - 1.
 * When to use it rather than gw_calc_witness_batch: for batches too small to fill the throughput kernel, where each
 * of its lanes walks the whole graph alone (a server answering a few to a few hundred concurrent requests).  Every
 * wave of one set per SM (148 on a B200) takes about one single-witness time.  Measured on a B200 at 1000 W (DESIGN.md
 * section 5g), device buffers: authV2 17.2 ms for 1 .. 148 sets against 85 ms on gw_calc_witness_batch, faster up to
 * about 740 sets; authV2_32_32 up to about 590; Poseidon(4) up to about 400.  Above that gw_calc_witness_batch is
 * faster.  Fails like gw_calc_witness_latency ("latency plan: graph is too wide ...") when the graph does not fit the
 * latency kernels; there is no fallback. */
int gw_calc_witness_latency_batch(gw_graph_t *graph, int first_device, int n_gpus, const uint8_t *inputs, size_t n_sets,
                                  uint8_t *witness, uint32_t *flags, gw_status_t *status);
/* the same on device buffers on `device`; ordered on cuda_stream (NULL = default stream); returns when the rows are
 * complete (the Boolean-graph fallback and the watchdog need a readback, as in gw_inputs_parse_batch_device) */
int gw_calc_witness_latency_batch_device(gw_graph_t *graph, int device, const void *d_inputs, size_t n_sets,
                                         void *d_witness, uint32_t *d_flags, void *cuda_stream, gw_status_t *status);

/* ---- batch input path (SURVEY 8f-1: replaces deserialize_inputs + populate_inputs, src/lib.rs:154-247, for many
 * input sets).  `text` is JSON Lines (one inputs object per non-empty line) or one top-level JSON array of such
 * objects; it is parsed by n_threads host threads (0 = all) into *inputs = a malloc'ed n_sets x n_inputs x 32 B
 * buffer in the layout gw_calc_witness_batch takes (caller frees).  Per-record semantics and error texts are those
 * of gw_calc_witness; the error message names the 1-based record. */
int gw_inputs_parse_batch(const gw_graph_t *graph, const char *text, size_t text_len, int n_threads,
                          uint8_t **inputs, size_t *n_sets, gw_status_t *status);

/* the same parse on CUDA device `device`: `text` (host memory, pageable or pinned; pinned copies faster) is copied
 * up once and split and parsed there; row r (n_inputs x 32 B) goes to d_inputs + r * n_inputs * 32, the layout
 * gw_calc_witness_batch_device reads.  *n_sets and the rows are byte-identical to gw_inputs_parse_batch, and so is
 * the error text.  Records outside the plain grammar (string escapes, '_' in numbers, repeated keys, "", errors) are
 * parsed by the host from the same text.  More than max_sets records is an error that leaves *n_sets = the count and
 * writes no row; max_sets = 0 with d_inputs = NULL only counts.  The work is ordered on `cuda_stream` (a cudaStream_t,
 * NULL = default stream); the call returns when the rows are complete, and later work on that stream sees them. */
int gw_inputs_parse_batch_device(const gw_graph_t *graph, int device, const char *text, size_t text_len,
                                 void *d_inputs, size_t max_sets, size_t *n_sets, void *cuda_stream,
                                 gw_status_t *status);

/* ---- batch output path (SURVEY 8f-2) ----
 * .wtns framing: like gw_calc_witness_batch, but set i is delivered as a complete .wtns file image
 * (wtns_from_witness, src/lib.rs:114-123: 76-byte header + n_witness x 32 B) at files + i * file_pitch;
 * file_pitch >= gw_wtns_file_size(graph) (bytes between consecutive images; pad as you like).  The payload rows
 * are placed by the device-to-host DMA itself (pitched copy), the headers are written by the host. */
size_t gw_wtns_file_size(const gw_graph_t *graph);
int gw_calc_witness_batch_wtns(gw_graph_t *graph, const uint8_t *inputs, size_t n_sets, uint8_t *files, size_t file_pitch,
                               uint32_t *flags, int n_gpus, gw_status_t *status);
/* Selected signals only (e.g. the public outputs): a new graph handle whose witness consists of the given witness
 * positions of `graph`, in the given order (repeats allowed).  Everything the selection does not depend on is dead
 * code for the device program, and only n_positions x 32 B per set cross PCIe.  All entry points work on the result;
 * free it with gw_graph_free. */
int gw_graph_select(const gw_graph_t *graph, const uint32_t *positions, size_t n_positions, gw_graph_t **selected,
                    gw_status_t *status);

/* Streaming (SURVEY 8f-2 "streaming D2H"): like gw_calc_witness_batch_on, but the witnesses are handed to `fn` chunk by
 * chunk as they land in a ring of three pinned host buffers per GPU that the library owns, so a batch whose witnesses
 * do not fit host memory (262 144 authV2 input sets = 806 GB) runs end to end at its real size.  `fn` is called with
 *   rows  : n_sets x row_bytes bytes (row_bytes = n_witness x 32), the witnesses of input sets first_set .. first_set + n_sets - 1,
 *   flags : n_sets x uint32 (the per-set bits of gw_calc_witness_batch),
 * valid only until it returns; returning nonzero stops the stream (the call then fails with an error).  One worker
 * thread per GPU calls it: chunks of one GPU arrive in order, chunks of different GPUs may arrive concurrently.
 * While `fn` looks at chunk k, chunk k + 1 is being copied and chunk k + 2 computed.  chunk_sets = 0 lets the library
 * choose (GW_STREAM_CHUNK_MB of pinned memory per ring slot, default 8192).  The worker threads are pinned to the CPUs of
 * their GPU's NUMA node before the ring is allocated (GW_NUMA=0 turns that off). */
typedef int (*gw_witness_chunk_fn)(void *user, int device, size_t first_set, size_t n_sets, const uint8_t *rows,
                                   size_t row_bytes, const uint32_t *flags);
int gw_calc_witness_batch_stream(gw_graph_t *graph, int first_device, int n_gpus, const uint8_t *inputs, size_t n_sets,
                                 size_t chunk_sets, gw_witness_chunk_fn fn, void *user, gw_status_t *status);

/* ---- R1CS check (the `snarkjs wtns check` step) ----
 * A graph has no constraints: an input set that violates the circuit (a bad signature, a stale Merkle root) still gets a
 * witness.  These calls check witnesses against the circuit's iden3 .r1cs file (version 1, as circom writes it) on the
 * GPU.  Wire i of the R1CS is witness position i, so n_wires == gw_graph_info_t.n_witness for the graph of the same
 * circuit.  A row passes when <A_k,w> * <B_k,w> == <C_k,w> (mod M) for every constraint k; a witness value >= M fails
 * the first constraint that reads it.  first_failed[r] receives the lowest violated constraint of row r, or GW_R1CS_OK. */
typedef struct gw_r1cs gw_r1cs_t;

typedef struct {
  uint32_t n_wires;       /* wires = witness length */
  uint32_t n_pub_out;     /* public outputs (wires 1 .. n_pub_out) */
  uint32_t n_pub_in;      /* public inputs (after the outputs) */
  uint32_t n_prv_in;      /* private inputs */
  uint32_t n_constraints;
  uint32_t n_consts;      /* distinct coefficients other than 1 and M - 1 (the device's constant table) */
  uint64_t n_labels;
  uint64_t n_terms;       /* compiled terms (zero coefficients dropped): 32-byte witness reads per row */
  uint64_t n_mac_terms;   /* terms with a coefficient other than 1 and M - 1: one 256 x 256-bit product each */
  uint64_t n_chunks;      /* Montgomery reductions: linear combinations are cut into chunks the accumulator can hold */
} gw_r1cs_info_t;

#define GW_R1CS_OK 0xFFFFFFFFu

/* parses and compiles an .r1cs file (no GPU needed).  Rejected with a message: bad magic, version != 1, missing header
 * or constraints section, truncated file or section, a section longer than its content, n8 != 32, a prime other than
 * BN254's, wire ids >= n_wires, custom-gate sections (4, 5).  Coefficients >= M are reduced mod M. */
int gw_r1cs_load(const void *data, size_t len, gw_r1cs_t **r1cs, gw_status_t *status);
void gw_r1cs_free(gw_r1cs_t *r1cs);
int gw_r1cs_info(const gw_r1cs_t *r1cs, gw_r1cs_info_t *info);
/* HOST rows: row r (n_wires x 32 B, canonical little-endian) at witness + r * row_pitch (row_pitch >= n_wires x 32;
 * 0 = dense).  With row_pitch = gw_wtns_file_size(graph) and witness = files + 76, the .wtns images of
 * gw_calc_witness_batch_wtns are checked in place.  The rows are split into n_gpus contiguous shards, one per device. */
int gw_r1cs_check_batch(gw_r1cs_t *r1cs, const uint8_t *witness, size_t n_sets, size_t row_pitch, uint32_t *first_failed,
                        int n_gpus, gw_status_t *status);
/* DEVICE rows on CUDA device `device` (d_witness and row_pitch 16-byte aligned; row_pitch 0 = dense), d_first_failed on
 * the same device; enqueued on `cuda_stream` (NULL = default stream) and asynchronous with respect to the host: what a
 * GPU prover pipeline calls after gw_calc_witness_batch_device on the same stream. */
int gw_r1cs_check_batch_device(gw_r1cs_t *r1cs, int device, const void *d_witness, size_t n_sets, size_t row_pitch,
                               uint32_t *d_first_failed, void *cuda_stream, gw_status_t *status);
/* gw_calc_witness_batch_on and the check in one pass: every chunk's witness rows are checked on the device right after
 * they are computed.  witness may be NULL: then only flags (optional) and first_failed cross PCIe.  Fails when
 * graph.n_witness != r1cs.n_wires. */
int gw_calc_witness_batch_check(gw_graph_t *graph, gw_r1cs_t *r1cs, int first_device, int n_gpus, const uint8_t *inputs,
                                size_t n_sets, uint8_t *witness, uint32_t *flags, uint32_t *first_failed,
                                gw_status_t *status);

/* ---- A, B and C of witness rows (the witness-dependent product of a prover, snarkjs / rapidsnark `buildABC`) ----
 * For every constraint k of row w: a_k = <A_k,w>, b_k = <B_k,w>, c_k = <C_k,w> (mod M), 32 bytes each, canonical
 * little-endian.  Output row = A[0..n) | B[0..n) | C[0..n).  A witness value >= M is reduced mod M before it enters a
 * linear combination.  first_failed (optional, may be NULL) receives the verdicts of gw_r1cs_check_batch, computed in
 * the same pass.
 *   options = 0                   n = n_constraints.
 *   options = GW_R1CS_ABC_GROTH16 the domain of a Groth16 prover (snarkjs zkey setup, read by rapidsnark): n = the
 *                                 smallest power of two >= n_constraints + n_pub + 1 (n_pub = n_pub_out + n_pub_in);
 *                                 entry n_constraints + s, s = 0 .. n_pub, has A = w_s and B = C = 0; the rest is 0. */
#define GW_R1CS_ABC_GROTH16 1u
/* entries per vector of one row: n_constraints, or with GW_R1CS_ABC_GROTH16 the power of two above; 0 for unknown
 * options or when the public signals do not fit the wires */
uint64_t gw_r1cs_abc_len(const gw_r1cs_t *r1cs, uint32_t options);
/* HOST rows (as gw_r1cs_check_batch: row_pitch 0 = dense, .wtns images in place with witness = files + 76);
 * abc: row r at abc + r * abc_pitch, abc_pitch >= 3 * n * 32 (0 = dense); bytes past 3 * n * 32 are not written;
 * first_failed optional; sharded over n_gpus devices.  n_sets = 0 does nothing. */
int gw_r1cs_abc_batch(gw_r1cs_t *r1cs, const uint8_t *witness, size_t n_sets, size_t row_pitch, uint8_t *abc,
                      size_t abc_pitch, uint32_t options, uint32_t *first_failed, int n_gpus, gw_status_t *status);
/* DEVICE buffers on `device` (16-byte aligned, pitches multiples of 16), asynchronous on cuda_stream (NULL = default
 * stream): composes with gw_calc_witness_batch_device on the same stream */
int gw_r1cs_abc_batch_device(gw_r1cs_t *r1cs, int device, const void *d_witness, size_t n_sets, size_t row_pitch,
                             void *d_abc, size_t abc_pitch, uint32_t options, uint32_t *d_first_failed,
                             void *cuda_stream, gw_status_t *status);

/* ---- Groth16 quotient evaluations and batched NTTs over the BN254 scalar field (M - 1 = 2^28 t) ----
 * w_28 = 5^t mod M (ffjavascript Fr.w[28], rapidsnark FFT); for n = 2^k: w_n = w_28^(2^(28 - k)), g = w_2n.
 * gw_fr_ntt_batch_device: in place, natural order in and out; vector v at d_data + v * pitch (pitch 0 = dense, else
 * >= n * 32 and a multiple of 16; d_data 16-byte aligned); inputs are any 256-bit values (reduced mod M), outputs
 * canonical 32-byte little-endian.  0 <= log_n <= 24.  Asynchronous on cuda_stream (NULL = default stream).
 *   flags 0                              y_j = sum_i x_i w_n^(ij)
 *   GW_NTT_INVERSE                       x_i = n^-1 sum_j y_j w_n^(-ij)
 *   GW_NTT_COSET                         y_j = sum_i x_i (g w_n^j)^i   (the input is multiplied by g^i first)
 *   GW_NTT_COSET | GW_NTT_INVERSE        the exact inverse of the coset transform (output i multiplied by g^-i)
 * n_vectors = 0 does nothing. */
#define GW_NTT_INVERSE 1u
#define GW_NTT_COSET 2u
int gw_fr_ntt_batch_device(int device, void *d_data, size_t n_vectors, uint32_t log_n, size_t pitch, uint32_t flags,
                           void *cuda_stream, gw_status_t *status);
/* h of every witness row (snarkjs groth16_prove joinABC, rapidsnark's vector before the H multi-scalar
 * multiplication): with n = gw_r1cs_abc_len(r1cs, GW_R1CS_ABC_GROTH16) and A, B, C the Groth16-layout vectors of
 * gw_r1cs_abc_batch, X_odd = the coset transform (GW_NTT_COSET) of the inverse transform (GW_NTT_INVERSE) of X and
 * h_i = A_odd[i] * B_odd[i] - C_odd[i] (mod M), i = 0 .. n - 1, 32 bytes each, canonical.  n > 2^24 is rejected.
 * first_failed (optional) receives the verdicts of gw_r1cs_check_batch from the same pass.
 * HOST rows as gw_r1cs_abc_batch (row_pitch 0 = dense, .wtns images in place with witness = files + 76); h row r at
 * h + r * h_pitch, h_pitch >= n * 32 (0 = dense); sharded over n_gpus devices.  n_sets = 0 does nothing. */
int gw_r1cs_quotient_batch(gw_r1cs_t *r1cs, const uint8_t *witness, size_t n_sets, size_t row_pitch, uint8_t *h,
                           size_t h_pitch, uint32_t *first_failed, int n_gpus, gw_status_t *status);
/* DEVICE buffers on `device` (16-byte aligned, pitches multiples of 16), asynchronous on cuda_stream: work row r at
 * d_work + r * work_pitch, work_pitch >= 3 * n * 32 (0 = dense); h is left in the first n * 32 bytes of each work row,
 * the rest of the row is scratch.  Composes with gw_calc_witness_batch_device on the same stream. */
int gw_r1cs_quotient_batch_device(gw_r1cs_t *r1cs, int device, const void *d_witness, size_t n_sets, size_t row_pitch,
                                  void *d_work, size_t work_pitch, uint32_t *d_first_failed, void *cuda_stream,
                                  gw_status_t *status);

/* CUDA device used by the single-witness entry points gw_calc_witness / gw_graph_calc_witness (default: the GW_DEVICE
 * environment variable, else device 0 of CUDA_VISIBLE_DEVICES).  Returns 1 if the device does not exist. */
int gw_set_device(int device);

/* writes the 76-byte .wtns header for n_witness values (src/lib.rs:114-123) */
void gw_wtns_header(uint32_t n_witness, uint8_t *dst76);

/* diagnostics */
int gw_device_count(void);
/* integer-pipe microbenchmark: executed multiply-add instructions per second on `device`;
 * which = 0 IMAD.WIDE.U32 carry rows (32x32+64, the form the field multiplier uses), 1 mad.lo.u32,
 * 2 mad.hi.u32, 3 add.u32 */
double gw_microbench_imad(int device, int which);

#ifdef __cplusplus
}
#endif

#endif /* RUST_GRAPH_WITNESS_H */
