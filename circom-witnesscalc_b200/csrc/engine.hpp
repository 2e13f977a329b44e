// A loaded witness graph: parsed, compiled to a device plan once, uploaded lazily per GPU.
// This is the persistent state the reference does not have (it re-parses the graph on every
// calc_witness call, /root/reference/src/lib.rs:129-130).
#pragma once
#include <atomic>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <string>

#include "bitplan.hpp"
#include "graph.hpp"
#include "plan.hpp"
#include "r1cs.hpp"

namespace gw {

class Engine {
 public:
  Engine(const uint8_t* graph_data, size_t len);
  explicit Engine(Graph g);     // an already parsed graph (gw_graph_select: same nodes, a subset of the witness)
  ~Engine();
  Engine(const Engine&) = delete;

  Graph graph;
  Plan plan;
  BitPlan bit_plan;           // bit-sliced plan (bitplan.hpp); used by every batch launch when eligible (GW_BITSLICE=0: never)
  std::atomic<bool> bit_disabled{false};   // set when most input sets of a launch broke the bit contract (engine.cu: launch)
  int max_threads = 512;      // upper bound of threads per CTA (GW_THREADS); one persistent CTA per SM
  int threads_for(size_t B, int sms, int t_max) const;
  int device_max_threads(int device);   // threads per CTA (= input sets per SM and wave) the device allows for this plan

  // inputs/witness resident on `device`: inputs [B][I][32 B LE], witness [B][W][32 B LE]; asynchronous on `stream`
  void run_device(int device, const void* d_inputs, size_t B, void* d_witness, uint32_t* d_status, void* stream);
  // host buffers; shards the batch over n_gpus devices starting at first_device (no collective)
  // witness row r is written at witness + r * out_pitch (out_pitch >= W * 32 bytes; 0 = dense rows): with a pitch of
  // wtns_size(W) rounded up and witness pointing WTNS_HEADER_BYTES into the first row, every row becomes a complete
  // .wtns file image once the caller has written the 76-byte headers (the DMA engine does the framing).
  // With `check`, every chunk's rows are also checked against that R1CS on the device (first_failed[r] = lowest violated
  // constraint of set r, or R1CS_OK), and witness may be null: then no witness row is copied to the host.
  // With `latency`, the chunks run on the latency kernels (run_latency_device) instead of the throughput kernel.
  void run_host(const uint8_t* inputs, size_t B, uint8_t* witness, uint32_t* status, int n_gpus, int first_device, size_t out_pitch = 0,
                R1cs* check = nullptr, uint32_t* first_failed = nullptr, bool latency = false);
  // Streaming output path: chunks of witness rows are handed to `fn` from a pinned ring as they land (one worker
  // thread per GPU; fn(device, first_set, n_sets, rows, row_bytes, flags) returns nonzero to stop).  The memory
  // is only valid during the call.  chunk_sets = 0 picks the chunk size.
  typedef std::function<int(int, size_t, size_t, const uint8_t*, size_t, const uint32_t*)> ChunkFn;
  void run_stream(const uint8_t* inputs, size_t B, int n_gpus, int first_device, size_t chunk_sets, const ChunkFn& fn);
  // single witness, latency mode (one CTA, intra-level node parallelism); host buffers
  void run_latency(int device, const uint8_t* inputs, uint8_t* witness, uint32_t* status, float* kernel_ms);
  // run_latency for B input sets resident on `device`, one latency CTA per set (as many at once as the device holds);
  // ordered on `stream`, returns when the rows are complete
  void run_latency_device(int device, const void* d_inputs, size_t B, void* d_witness, uint32_t* d_status, void* stream);
  // a plan without LUTs is pure wiring: worth it only when field inputs are taken apart into bits (Num2Bits of a field element)
  bool use_bit_path() const { return bit_plan.eligible && (bit_plan.n_luts > 0 || bit_plan.has_field_inputs); }
  bool bit_path_active() const { return use_bit_path() && !bit_disabled.load(); }
  LatencyPlan lat_plan;
  bool lat_ready = false;
  std::string lat_error;      // why the latency plan could not be built (remembered: the compile is not repeated per call)

 private:
  struct Dev;
  Dev* dev(int device);
  void launch(Dev* d, const void* d_inputs, size_t B, void* d_witness, uint32_t* d_status, void* stream);
  void launch_bit(Dev* d, const void* d_inputs, size_t B, void* d_witness, uint32_t* d_status, void* stream);
  const LatencyPlan& latency_plan(Dev* d);
  bool latency_bit(Dev* d) const;
  size_t latency_wave(Dev* d);
  void latency_kernels(Dev* d, const void* d_inputs, size_t n, const uint32_t* row_map, void* d_witness, uint32_t* d_status, void* stream);
  void latency_launch(Dev* d, const void* d_inputs, size_t B, void* d_witness, uint32_t* d_status, void* stream);
  void latency_arm(Dev* d, void* stream);
  void latency_check(Dev* d);
  void ensure_staging(Dev* d, size_t chunk);
  void stream_on(int device, const uint8_t* inputs, size_t B, size_t first_set, size_t chunk_req, const ChunkFn& fn);
  void run_host_on(int device, const uint8_t* inputs, size_t B, uint8_t* witness, uint32_t* status, size_t out_pitch, R1cs* check,
                   uint32_t* first_failed, bool latency);
  void init_plan();
  std::map<int, std::unique_ptr<Dev>> devs;
  std::mutex mu;
};

double imad_microbench(int device, int which);

}  // namespace gw
