// extern "C" boundary: include/graph_witness.h.  Replaces /root/reference/src/lib.rs:28-111
// (prepare_status, gw_calc_witness).  Nothing may unwind across this boundary (the reference's
// unwrap()/panic!s would be UB here, lib.rs:130,160,196): every entry point catches everything.
#include "../../include/graph_witness.h"

#include <string.h>

#include <atomic>
#include <list>
#include <memory>
#include <mutex>

#include "cuda_util.hpp"
#include "engine.hpp"
#include "inputs.hpp"
#include "ntt.hpp"
#include "wtns.hpp"

using namespace gw;

struct gw_graph {
  std::unique_ptr<Engine> engine;
  std::vector<std::string> input_names;
  // device input parser (key tables and scratch per device), made by the first gw_inputs_parse_batch_device
  mutable std::unique_ptr<DeviceInputs> dev_inputs;
  mutable std::mutex dev_inputs_mu;
};

struct gw_r1cs {
  std::unique_ptr<R1cs> r1cs;
};

static void set_status(const gw_status_t* status_c, GW_ERROR_CODE code, const char* msg) {   // lib.rs:28-38
  gw_status_t* status = const_cast<gw_status_t*>(status_c);
  if (!status) return;
  status->code = code;
  status->error_msg = nullptr;
  if (msg) {
    size_t n = strlen(msg);
    status->error_msg = (char*)malloc(n + 1);
    if (status->error_msg) memcpy(status->error_msg, msg, n + 1);
  }
}

template <typename F> static int guarded(const gw_status_t* status, F&& f) {
  try { f(); set_status(status, OK, nullptr); return 0; }
  catch (const std::exception& e) { set_status(status, ERROR, e.what()); return 1; }
  catch (...) { set_status(status, ERROR, "unknown error"); return 1; }
}

static const char* const RANGE_ERROR = "device range exceeds the visible CUDA devices";   // host entry points with a first_device
static const char* const N_GPUS_ERROR = "n_gpus exceeds the number of visible CUDA devices";   // host entry points that start at device 0

// The devices [first_device, first_device + n_gpus) of a host entry point (n_gpus < 1: one device); range_error is the
// message of the entry point's family.  Returns n_gpus.
static int check_devices(int first_device, int n_gpus, const char* range_error) {
  const int ndev = cuda_device_count();
  if (ndev == 0) throw Error(NO_DEVICE_ERROR);
  if (n_gpus < 1) n_gpus = 1;
  if (first_device < 0 || first_device + n_gpus > ndev) throw Error(range_error);
  return n_gpus;
}

static int single_device();
static void calc_one(Engine& eng, const char* json, void** wtns_data, size_t* wtns_len) {
  InputList in = deserialize_inputs(json, strlen(json));
  std::vector<U256> buf = build_inputs_buffer(eng.graph, in);
  const uint32_t W = eng.plan.n_witness;
  const int dev = single_device();
  size_t n = wtns_size(W);
  uint8_t* out = (uint8_t*)malloc(n);
  if (!out) throw Error("Failed to allocate memory for wtns_data");
  try {
    wtns_write_header(out, W);
    // a single witness goes through the latency-mode kernel (intra-level node parallelism) unless
    // GW_SINGLE_MODE=batch asks for the throughput kernel with a batch of one
    const char* mode = getenv("GW_SINGLE_MODE");
    if (mode && !strcmp(mode, "batch")) eng.run_host((const uint8_t*)buf.data(), 1, out + WTNS_HEADER_BYTES, nullptr, 1, dev);
    else {
      // a graph whose live values do not fit the latency kernel's shared-memory value file still gets its witness from
      // the GPU: the throughput kernel with a batch of one
      try { eng.run_latency(dev, (const uint8_t*)buf.data(), out + WTNS_HEADER_BYTES, nullptr, nullptr); }
      catch (const Error& e) {
        if (strncmp(e.what(), "latency plan:", 13) != 0) throw;
        eng.run_host((const uint8_t*)buf.data(), 1, out + WTNS_HEADER_BYTES, nullptr, 1, dev);
      }
    }
  } catch (...) { free(out); throw; }
  *wtns_data = out; *wtns_len = n;
}

// gw_calc_witness is stateless for the caller; parsed graphs are kept in a small cache keyed by content.  A hit is
// confirmed by comparing the bytes (the hash only narrows the search), and engines are built outside the lock.
struct CacheEntry { uint64_t hash; std::vector<uint8_t> bytes; std::shared_ptr<Engine> engine; };
static std::mutex g_cache_mu;
static std::list<CacheEntry> g_cache;
static std::shared_ptr<Engine> cached_engine(const uint8_t* data, size_t len) {
  uint64_t h = 1469598103934665603ull;
  for (size_t i = 0; i < len; i++) { h ^= data[i]; h *= 1099511628211ull; }
  auto lookup = [&]() -> std::shared_ptr<Engine> {
    for (auto it = g_cache.begin(); it != g_cache.end(); ++it)
      if (it->hash == h && it->bytes.size() == len && memcmp(it->bytes.data(), data, len) == 0) { g_cache.splice(g_cache.begin(), g_cache, it); return g_cache.front().engine; }
    return nullptr;
  };
  {
    std::lock_guard<std::mutex> lk(g_cache_mu);
    if (std::shared_ptr<Engine> e = lookup()) return e;
  }
  std::shared_ptr<Engine> e(new Engine(data, len));         // parse + plan compilation: other callers are not held up
  std::lock_guard<std::mutex> lk(g_cache_mu);
  if (std::shared_ptr<Engine> other = lookup()) return other;   // somebody else built the same graph meanwhile
  g_cache.push_front(CacheEntry{h, std::vector<uint8_t>(data, data + len), e});
  if (g_cache.size() > 4) g_cache.pop_back();
  return e;
}

// device of the single-witness entry points (gw_calc_witness, gw_graph_calc_witness): gw_set_device, else GW_DEVICE, else 0
static std::atomic<int> g_device{-1};
static int single_device() {
  int d = g_device.load();
  if (d >= 0) return d;
  const char* s = getenv("GW_DEVICE");
  return (s && *s) ? atoi(s) : 0;
}

extern "C" {

int gw_calc_witness(const char* inputs, const void* graph_data, const size_t graph_data_len, void** wtns_data,
                    size_t* wtns_len, const gw_status_t* status) {
  if (!inputs) { set_status(status, ERROR, "inputs is null"); return 1; }             // lib.rs:51-54
  if (!graph_data) { set_status(status, ERROR, "graph_data is null"); return 1; }     // lib.rs:56-59
  if (graph_data_len == 0) { set_status(status, ERROR, "graph_data_len is 0"); return 1; }   // lib.rs:61-64
  if (!wtns_data || !wtns_len) { set_status(status, ERROR, "wtns_data or wtns_len is null"); return 1; }
  return guarded(status, [&]() {
    std::shared_ptr<Engine> e = cached_engine((const uint8_t*)graph_data, graph_data_len);
    calc_one(*e, inputs, wtns_data, wtns_len);
  });
}

int gw_graph_load(const void* graph_data, size_t graph_data_len, gw_graph_t** graph, gw_status_t* status) {
  if (!graph_data || graph_data_len == 0 || !graph) { set_status(status, ERROR, "graph_data is null or empty"); return 1; }
  return guarded(status, [&]() {
    std::unique_ptr<gw_graph> g(new gw_graph());
    g->engine.reset(new Engine((const uint8_t*)graph_data, graph_data_len));
    for (auto& kv : g->engine->graph.inputs) g->input_names.push_back(kv.first);
    *graph = g.release();
  });
}

void gw_graph_free(gw_graph_t* graph) { delete graph; }

int gw_graph_info(const gw_graph_t* graph, gw_graph_info_t* info) {
  if (!graph || !info) return 1;
  const Plan& p = graph->engine->plan;
  memset(info, 0, sizeof *info);
  info->n_nodes = p.stats.graph_nodes; info->n_ops = p.stats.graph_ops;
  info->n_inputs = p.n_inputs; info->n_witness = p.n_witness;
  info->n_input_signals = (uint32_t)graph->input_names.size();
  info->n_instrs = (uint32_t)p.stats.instrs; info->n_regs = p.n_regs; info->n_spill = p.n_spill + (p.n_spill_narrow + 3) / 4;   /* 32-byte slot equivalents */
  info->n_mul = p.stats.mul_nodes; info->n_div = p.stats.div_nodes;
  info->n_spill_ld = p.stats.spill_ld; info->n_spill_st = p.stats.spill_st;
  info->n_slots = (uint32_t)p.stats.slots; info->n_dot = (uint32_t)p.stats.op_count[OP_DOT];
  info->n_dot_mac = (uint32_t)p.stats.dot_terms[T_MAC];
  info->n_mul_instr = (uint32_t)(p.stats.op_count[OP_MUL] + p.stats.op_count[OP_SQR]);
  info->n_inversions = (uint32_t)p.stats.inversions;
  info->threads = (uint32_t)graph->engine->max_threads; info->sets_per_thread = 1;
  info->n_narrow_instr = (uint32_t)p.stats.narrow_instrs;
  const BitPlan& bp = graph->engine->bit_plan;
  info->bit_eligible = graph->engine->bit_path_active() ? 1u : 0u;
  info->bit_luts = (uint32_t)bp.n_luts; info->bit_steps = bp.n_steps; info->bit_wide = (uint32_t)(bp.wide.size() / 3);
  return 0;
}

int gw_graph_input_signal(const gw_graph_t* graph, uint32_t i, const char** name, uint32_t* offset, uint32_t* len) {
  if (!graph || i >= graph->input_names.size()) return 1;
  auto it = graph->engine->graph.inputs.find(graph->input_names[i]);
  if (name) *name = graph->input_names[i].c_str();
  if (offset) *offset = it->second.first;
  if (len) *len = it->second.second;
  return 0;
}

int gw_graph_calc_witness(gw_graph_t* graph, const char* inputs_json, void** wtns_data, size_t* wtns_len, gw_status_t* status) {
  if (!graph || !inputs_json || !wtns_data || !wtns_len) { set_status(status, ERROR, "null argument"); return 1; }
  return guarded(status, [&]() { calc_one(*graph->engine, inputs_json, wtns_data, wtns_len); });
}

int gw_calc_witness_batch_on(gw_graph_t* graph, int first_device, const uint8_t* inputs, size_t n_sets, uint8_t* witness,
                             uint32_t* flags, int n_gpus, gw_status_t* status) {
  if (!graph || (n_sets && (!inputs || !witness))) { set_status(status, ERROR, "null argument"); return 1; }
  return guarded(status, [&]() {
    n_gpus = check_devices(first_device, n_gpus, RANGE_ERROR);
    graph->engine->run_host(inputs, n_sets, witness, flags, n_gpus, first_device);
  });
}

int gw_calc_witness_batch(gw_graph_t* graph, const uint8_t* inputs, size_t n_sets, uint8_t* witness, uint32_t* flags,
                          int n_gpus, gw_status_t* status) {
  if (graph && n_gpus > cuda_device_count() && cuda_device_count() > 0) { set_status(status, ERROR, N_GPUS_ERROR); return 1; }
  return gw_calc_witness_batch_on(graph, 0, inputs, n_sets, witness, flags, n_gpus, status);
}

int gw_calc_witness_batch_device(gw_graph_t* graph, int device, const void* d_inputs, size_t n_sets, void* d_witness,
                                 uint32_t* d_flags, void* cuda_stream, gw_status_t* status) {
  if (!graph || (n_sets && (!d_inputs || !d_witness))) { set_status(status, ERROR, "null argument"); return 1; }
  return guarded(status, [&]() { graph->engine->run_device(device, d_inputs, n_sets, d_witness, d_flags, cuda_stream); });
}

int gw_calc_witness_latency(gw_graph_t* graph, int device, const uint8_t* inputs, uint8_t* witness, uint32_t* flags,
                            float* kernel_ms, gw_status_t* status) {
  if (!graph || !inputs || !witness) { set_status(status, ERROR, "null argument"); return 1; }
  return guarded(status, [&]() { graph->engine->run_latency(device, inputs, witness, flags, kernel_ms); });
}

int gw_calc_witness_latency_batch(gw_graph_t* graph, int first_device, int n_gpus, const uint8_t* inputs, size_t n_sets,
                                  uint8_t* witness, uint32_t* flags, gw_status_t* status) {
  if (!graph || (n_sets && (!inputs || !witness))) { set_status(status, ERROR, "null argument"); return 1; }
  return guarded(status, [&]() {
    if (!n_sets) return;
    n_gpus = check_devices(first_device, n_gpus, RANGE_ERROR);
    graph->engine->run_host(inputs, n_sets, witness, flags, n_gpus, first_device, 0, nullptr, nullptr, true);
  });
}

int gw_calc_witness_latency_batch_device(gw_graph_t* graph, int device, const void* d_inputs, size_t n_sets, void* d_witness,
                                         uint32_t* d_flags, void* cuda_stream, gw_status_t* status) {
  if (!graph || (n_sets && (!d_inputs || !d_witness))) { set_status(status, ERROR, "null argument"); return 1; }
  return guarded(status, [&]() { graph->engine->run_latency_device(device, d_inputs, n_sets, d_witness, d_flags, cuda_stream); });
}

int gw_inputs_parse_batch(const gw_graph_t* graph, const char* text, size_t text_len, int n_threads, uint8_t** inputs,
                          size_t* n_sets, gw_status_t* status) {
  if (!graph || !text || !inputs || !n_sets) { set_status(status, ERROR, "null argument"); return 1; }
  return guarded(status, [&]() {
    U256* rows = nullptr;
    size_t n = parse_inputs_batch(graph->engine->graph, text, text_len, n_threads, &rows);
    *inputs = (uint8_t*)rows; *n_sets = n;
  });
}

int gw_inputs_parse_batch_device(const gw_graph_t* graph, int device, const char* text, size_t text_len, void* d_inputs,
                                 size_t max_sets, size_t* n_sets, void* cuda_stream, gw_status_t* status) {
  if (!graph || !n_sets || (text_len && !text) || (max_sets && !d_inputs)) { set_status(status, ERROR, "null argument"); return 1; }
  *n_sets = 0;
  return guarded(status, [&]() {
    DeviceInputs* p;
    {
      std::lock_guard<std::mutex> lk(graph->dev_inputs_mu);
      if (!graph->dev_inputs) graph->dev_inputs.reset(new DeviceInputs(graph->engine->graph));
      p = graph->dev_inputs.get();
    }
    p->parse(device, text, text_len, d_inputs, max_sets, cuda_stream, n_sets);
  });
}

size_t gw_wtns_file_size(const gw_graph_t* graph) { return graph ? wtns_size(graph->engine->plan.n_witness) : 0; }

int gw_calc_witness_batch_wtns(gw_graph_t* graph, const uint8_t* inputs, size_t n_sets, uint8_t* files, size_t file_pitch,
                               uint32_t* flags, int n_gpus, gw_status_t* status) {
  if (!graph || (n_sets && (!inputs || !files))) { set_status(status, ERROR, "null argument"); return 1; }
  return guarded(status, [&]() {
    const uint32_t W = graph->engine->plan.n_witness;
    if (file_pitch < wtns_size(W)) throw Error("file_pitch is smaller than a .wtns file of this graph");
    n_gpus = check_devices(0, n_gpus, N_GPUS_ERROR);
    for (size_t i = 0; i < n_sets; i++) wtns_write_header(files + i * file_pitch, W);
    graph->engine->run_host(inputs, n_sets, files + WTNS_HEADER_BYTES, flags, n_gpus, 0, file_pitch);
  });
}

int gw_graph_select(const gw_graph_t* graph, const uint32_t* positions, size_t n_positions, gw_graph_t** selected,
                    gw_status_t* status) {
  if (!graph || !selected || (n_positions && !positions)) { set_status(status, ERROR, "null argument"); return 1; }
  return guarded(status, [&]() {
    Graph sub = graph->engine->graph;                       // same nodes, constants and input map
    const std::vector<uint32_t>& ws = graph->engine->graph.witness_signals;
    sub.witness_signals.clear();
    for (size_t i = 0; i < n_positions; i++) {
      if (positions[i] >= ws.size()) throw Error("witness position out of range");
      sub.witness_signals.push_back(ws[positions[i]]);
    }
    std::unique_ptr<gw_graph> g(new gw_graph());
    g->engine.reset(new Engine(std::move(sub)));
    g->input_names = graph->input_names;
    *selected = g.release();
  });
}

int gw_calc_witness_batch_stream(gw_graph_t* graph, int first_device, int n_gpus, const uint8_t* inputs, size_t n_sets,
                                 size_t chunk_sets, gw_witness_chunk_fn fn, void* user, gw_status_t* status) {
  if (!graph || !fn || (n_sets && !inputs)) { set_status(status, ERROR, "null argument"); return 1; }
  return guarded(status, [&]() {
    n_gpus = check_devices(first_device, n_gpus, RANGE_ERROR);
    graph->engine->run_stream(inputs, n_sets, n_gpus, first_device, chunk_sets,
                              [&](int device, size_t first, size_t n, const uint8_t* rows, size_t row_bytes, const uint32_t* flags) {
                                return fn(user, device, first, n, rows, row_bytes, flags);
                              });
  });
}

int gw_r1cs_load(const void* data, size_t len, gw_r1cs_t** r1cs, gw_status_t* status) {
  if (!data || !r1cs) { set_status(status, ERROR, "null argument"); return 1; }
  return guarded(status, [&]() {
    std::unique_ptr<gw_r1cs> r(new gw_r1cs());
    r->r1cs.reset(new R1cs((const uint8_t*)data, len));
    *r1cs = r.release();
  });
}

void gw_r1cs_free(gw_r1cs_t* r1cs) { delete r1cs; }

int gw_r1cs_info(const gw_r1cs_t* r1cs, gw_r1cs_info_t* info) {
  if (!r1cs || !info) return 1;
  const R1cs& r = *r1cs->r1cs;
  memset(info, 0, sizeof *info);
  info->n_wires = r.hdr.n_wires; info->n_pub_out = r.hdr.n_pub_out; info->n_pub_in = r.hdr.n_pub_in; info->n_prv_in = r.hdr.n_prv_in;
  info->n_constraints = r.hdr.n_constraints; info->n_consts = (uint32_t)r.prog.consts.size(); info->n_labels = r.hdr.n_labels;
  info->n_terms = r.prog.n_terms; info->n_mac_terms = r.prog.n_mac_terms; info->n_chunks = r.prog.n_chunks;
  return 0;
}

int gw_r1cs_check_batch(gw_r1cs_t* r1cs, const uint8_t* witness, size_t n_sets, size_t row_pitch, uint32_t* first_failed,
                        int n_gpus, gw_status_t* status) {
  if (!r1cs || (n_sets && (!witness || !first_failed))) { set_status(status, ERROR, "null argument"); return 1; }
  return guarded(status, [&]() {
    n_gpus = check_devices(0, n_gpus, N_GPUS_ERROR);
    r1cs->r1cs->check_host(witness, n_sets, row_pitch ? row_pitch : (size_t)r1cs->r1cs->hdr.n_wires * 32, first_failed, n_gpus, 0);
  });
}

int gw_r1cs_check_batch_device(gw_r1cs_t* r1cs, int device, const void* d_witness, size_t n_sets, size_t row_pitch,
                               uint32_t* d_first_failed, void* cuda_stream, gw_status_t* status) {
  if (!r1cs || (n_sets && (!d_witness || !d_first_failed))) { set_status(status, ERROR, "null argument"); return 1; }
  return guarded(status, [&]() {
    r1cs->r1cs->check_device(device, d_witness, n_sets, row_pitch ? row_pitch : (size_t)r1cs->r1cs->hdr.n_wires * 32, d_first_failed,
                             cuda_stream);
  });
}

uint64_t gw_r1cs_abc_len(const gw_r1cs_t* r1cs, uint32_t options) {
  if (!r1cs) return 0;
  try { return r1cs->r1cs->abc_len(options); } catch (...) { return 0; }
}

int gw_r1cs_abc_batch(gw_r1cs_t* r1cs, const uint8_t* witness, size_t n_sets, size_t row_pitch, uint8_t* abc, size_t abc_pitch,
                      uint32_t options, uint32_t* first_failed, int n_gpus, gw_status_t* status) {
  if (!r1cs || (n_sets && (!witness || !abc))) { set_status(status, ERROR, "null argument"); return 1; }
  return guarded(status, [&]() {
    R1cs& r = *r1cs->r1cs;
    if (!row_pitch) row_pitch = (size_t)r.hdr.n_wires * 32;
    if (!abc_pitch) abc_pitch = 3 * 32 * (size_t)r.abc_len(options);
    r.abc_row_bytes(row_pitch, abc_pitch, options, false);          // the arguments first: no device is touched
    if (!n_sets) return;
    n_gpus = check_devices(0, n_gpus, N_GPUS_ERROR);
    r.abc_host(witness, n_sets, row_pitch, abc, abc_pitch, options, first_failed, n_gpus, 0);
  });
}

int gw_r1cs_abc_batch_device(gw_r1cs_t* r1cs, int device, const void* d_witness, size_t n_sets, size_t row_pitch, void* d_abc,
                             size_t abc_pitch, uint32_t options, uint32_t* d_first_failed, void* cuda_stream, gw_status_t* status) {
  if (!r1cs || (n_sets && (!d_witness || !d_abc))) { set_status(status, ERROR, "null argument"); return 1; }
  return guarded(status, [&]() {
    R1cs& r = *r1cs->r1cs;
    if (!row_pitch) row_pitch = (size_t)r.hdr.n_wires * 32;
    if (!abc_pitch) abc_pitch = 3 * 32 * (size_t)r.abc_len(options);
    r.abc_device(device, d_witness, n_sets, row_pitch, d_abc, abc_pitch, options, d_first_failed, cuda_stream);
  });
}

int gw_fr_ntt_batch_device(int device, void* d_data, size_t n_vectors, uint32_t log_n, size_t pitch, uint32_t flags,
                           void* cuda_stream, gw_status_t* status) {
  if (n_vectors && !d_data) { set_status(status, ERROR, "null argument"); return 1; }
  return guarded(status, [&]() { ntt_batch_device(device, d_data, n_vectors, log_n, pitch, flags, cuda_stream); });
}

int gw_r1cs_quotient_batch(gw_r1cs_t* r1cs, const uint8_t* witness, size_t n_sets, size_t row_pitch, uint8_t* h, size_t h_pitch,
                           uint32_t* first_failed, int n_gpus, gw_status_t* status) {
  if (!r1cs || (n_sets && (!witness || !h))) { set_status(status, ERROR, "null argument"); return 1; }
  return guarded(status, [&]() {
    R1cs& r = *r1cs->r1cs;
    if (!row_pitch) row_pitch = (size_t)r.hdr.n_wires * 32;
    if (!h_pitch) h_pitch = 32 * (size_t)r.abc_len(GW_R1CS_ABC_GROTH16);
    r.quotient_log_n(row_pitch, h_pitch, false);                    // the arguments first: no device is touched
    if (!n_sets) return;
    n_gpus = check_devices(0, n_gpus, N_GPUS_ERROR);
    r.quotient_host(witness, n_sets, row_pitch, h, h_pitch, first_failed, n_gpus, 0);
  });
}

int gw_r1cs_quotient_batch_device(gw_r1cs_t* r1cs, int device, const void* d_witness, size_t n_sets, size_t row_pitch, void* d_work,
                                  size_t work_pitch, uint32_t* d_first_failed, void* cuda_stream, gw_status_t* status) {
  if (!r1cs || (n_sets && (!d_witness || !d_work))) { set_status(status, ERROR, "null argument"); return 1; }
  return guarded(status, [&]() {
    R1cs& r = *r1cs->r1cs;
    if (!row_pitch) row_pitch = (size_t)r.hdr.n_wires * 32;
    if (!work_pitch) work_pitch = 3 * 32 * (size_t)r.abc_len(GW_R1CS_ABC_GROTH16);
    r.quotient_device(device, d_witness, n_sets, row_pitch, d_work, work_pitch, d_first_failed, cuda_stream);
  });
}

int gw_calc_witness_batch_check(gw_graph_t* graph, gw_r1cs_t* r1cs, int first_device, int n_gpus, const uint8_t* inputs,
                                size_t n_sets, uint8_t* witness, uint32_t* flags, uint32_t* first_failed, gw_status_t* status) {
  if (!graph || !r1cs || (n_sets && (!inputs || !first_failed))) { set_status(status, ERROR, "null argument"); return 1; }
  return guarded(status, [&]() {
    const uint32_t W = graph->engine->plan.n_witness, n_wires = r1cs->r1cs->hdr.n_wires;
    if (W != n_wires)
      throw Error("the graph's witness has " + std::to_string(W) + " values but the R1CS has " + std::to_string(n_wires) + " wires");
    n_gpus = check_devices(first_device, n_gpus, RANGE_ERROR);
    graph->engine->run_host(inputs, n_sets, witness, flags, n_gpus, first_device, 0, r1cs->r1cs.get(), first_failed);
  });
}

int gw_set_device(int device) {
  if (device < 0 || device >= cuda_device_count()) return 1;
  g_device.store(device);
  return 0;
}

void gw_wtns_header(uint32_t n_witness, uint8_t* dst76) { wtns_write_header(dst76, n_witness); }

int gw_device_count(void) { return cuda_device_count(); }

double gw_microbench_imad(int device, int which) {
  try { return imad_microbench(device, which); } catch (...) { return -1.0; }
}

}  // extern "C"
