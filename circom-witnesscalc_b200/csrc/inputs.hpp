// Inputs JSON -> flat input buffer.
// Mirrors /root/reference/src/lib.rs:195-247 (deserialize_inputs), :154-181 (populate_inputs,
// get_inputs_buffer).  Errors the reference reports as Error::InputsUnmarshal /
// InputFieldNumberParseError keep their wording; cases where the reference panics (invalid JSON,
// unknown key, wrong length) are reported as gw::Error instead.
#pragma once
#include <memory>
#include <mutex>

#include "graph.hpp"

namespace gw {

typedef std::vector<std::pair<std::string, std::vector<U256>>> InputList;   // insertion order kept

InputList deserialize_inputs(const char* json, size_t len);
// buffer of g.inputs_size values, slot 0 = 1, unmentioned slots = 0 (lib.rs:177-181)
std::vector<U256> build_inputs_buffer(const Graph& g, const InputList& inputs);


// Batch input path (SURVEY 8f rank 1): a JSON Lines text (one inputs object per non-empty line; a single top-level
// JSON array of objects is accepted too) -> n_sets x inputs_size x 32 B packed little-endian rows, parsed by
// n_threads host threads (0 = hardware concurrency).  Every row goes through deserialize_inputs +
// build_inputs_buffer, so values, errors and missing-key behaviour are those of the single-witness path.
// Errors name the 1-based record.  *out_rows receives a malloc'ed buffer of n_sets * inputs_size values (caller frees;
// null after an error).
size_t parse_inputs_batch(const Graph& g, const char* text, size_t len, int n_threads, U256** out_rows);
// the record boundaries [first, second) of such a text; throws on an unterminated array or bytes after it
void split_records(const char* text, size_t len, std::vector<std::pair<size_t, size_t>>& rec);

// The same parse on a CUDA device (inputs.cu): the text is copied up once, split into records and parsed there, and
// row r is written to d_rows + r * inputs_size * 32.  Rows and errors are those of parse_inputs_batch: the device
// parser accepts only the plain grammar real inputs use and marks every other record, which the host then parses with
// deserialize_inputs + build_inputs_buffer.  Ordered on `stream`; returns when the rows are complete.  *n_sets receives
// the record count, also when there are more than max_sets records (an error: nothing is written then).
class DeviceInputs {
 public:
  explicit DeviceInputs(const Graph& g);
  ~DeviceInputs();
  DeviceInputs(const DeviceInputs&) = delete;
  void parse(int device, const char* text, size_t len, void* d_rows, size_t max_sets, void* stream, size_t* n_sets);
  struct Dev;

 private:
  Dev* dev(int device);
  const Graph& g;
  std::map<int, std::unique_ptr<Dev>> devs;
  std::mutex mu;
};

}  // namespace gw
