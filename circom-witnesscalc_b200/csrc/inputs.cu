// Batch input path on the device (gw_inputs_parse_batch_device): JSON Lines or one JSON array of input objects ->
// dense n_sets x inputs_size x 32 B rows in HBM, byte-identical to parse_inputs_batch (inputs.cpp).
//
// 1. Record split.  The text is cut into tiles of SPLIT_TILE bytes.  The string state of every byte comes from a
//    3-state transducer (JSON Lines: "no non-blank byte on this line yet" / "seen one"; array form: outside a string /
//    inside / after a backslash) whose per-byte maps are composed by a prefix scan, within a tile and then over the
//    tiles.  The array form adds a prefix sum of the bracket depth over the bytes outside strings.  A JSON Lines
//    record starts at the first non-blank byte of a line; an array record is a '{' at depth 1 and ends at the '}' that
//    brings the depth back to 1, as in split_records.  Split errors and odd layouts go to split_records on the host.
// 2. Record parse: one thread per record, for the grammar real inputs use (an object of "key": value members, keys
//    without escapes, values "<digits>", bare u64 integers or arrays of those, every key known, once, with the right
//    number of values).  Every other record is marked and parsed by the host, which also reports the lowest failing
//    record.  The device parser is only sound: what it accepts is what the host would produce.
#include "inputs.hpp"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <memory>

#include "cuda_util.hpp"

namespace gw {

namespace {

constexpr int SPLIT_THREADS = 256, SPLIT_BYTES = 64;                 // bytes per thread: four 16-byte loads
constexpr size_t SPLIT_TILE = (size_t)SPLIT_THREADS * SPLIT_BYTES;
constexpr int SCAN_THREADS = 1024, PARSE_THREADS = 128;
enum : uint32_t { FORM_LINES = 0, FORM_ARRAY = 1 };
enum : uint32_t { S_OUT = 0, S_IN = 1, S_ESC = 2 };                  // array-form string state
// summary words of one split: record starts and ends, the position of the byte that closes the array (~0: none) and
// 1 + the position of the last non-blank byte (0: none)
enum { SUM_STARTS = 0, SUM_ENDS = 1, SUM_CLOSE = 2, SUM_LAST = 3, SUM_MARKS = 4, SUM_ODD = 5, SUM_WORDS = 8 };

// a map of the 3 states, 2 bits per state
constexpr uint32_t FN_ID = 0u | 1u << 2 | 2u << 4;
__device__ __forceinline__ uint32_t fn_apply(uint32_t f, uint32_t s) { return (f >> (2 * s)) & 3u; }
struct FnThen {   // a first, then b
  __device__ __forceinline__ uint32_t operator()(uint32_t a, uint32_t b) const {
    return fn_apply(b, fn_apply(a, 0)) | fn_apply(b, fn_apply(a, 1)) << 2 | fn_apply(b, fn_apply(a, 2)) << 4;
  }
};
struct Add {
  template <typename T> __device__ __forceinline__ T operator()(T a, T b) const { return a + b; }
};

__device__ __forceinline__ bool is_blank(uint32_t c) { return c == ' ' || c == '\t' || c == '\r'; }
__device__ __forceinline__ bool is_ws(uint32_t c) { return is_blank(c) || c == '\n'; }

__device__ __forceinline__ uint32_t byte_fn(uint32_t form, uint32_t c) {
  if (form == FORM_LINES) {
    if (c == '\n') return 0;
    return is_blank(c) ? FN_ID : (1u | 1u << 2 | 1u << 4);
  }
  if (c == '"') return S_IN | S_OUT << 2 | S_IN << 4;
  if (c == '\\') return S_OUT | S_ESC << 2 | S_IN << 4;
  return S_OUT | S_IN << 2 | S_IN << 4;
}

// exclusive scan over the block (SPLIT_THREADS threads) of an associative, not necessarily commutative, operation
template <typename T, typename Op>
__device__ T block_scan(T v, T id, Op op, T* total) {
  __shared__ T warp_sum[SPLIT_THREADS / 32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  T inc = v;
  for (int o = 1; o < 32; o <<= 1) {
    const T u = __shfl_up_sync(0xFFFFFFFFu, inc, o);
    if (lane >= o) inc = op(u, inc);
  }
  T ex = __shfl_up_sync(0xFFFFFFFFu, inc, 1);
  if (lane == 0) ex = id;
  if (lane == 31) warp_sum[w] = inc;
  __syncthreads();
  T pre = id, all = id;
  for (int k = 0; k < SPLIT_THREADS / 32; k++) {
    if (k < w) pre = op(pre, warp_sum[k]);
    all = op(all, warp_sum[k]);
  }
  __syncthreads();                       // warp_sum is reused by the next scan
  *total = all;
  return op(pre, ex);
}

__device__ __forceinline__ uint32_t byte_of(const uint4* b, int k) {
  const uint4 q = b[k >> 4];
  const uint32_t w = (k & 8) ? ((k & 4) ? q.w : q.z) : ((k & 4) ? q.y : q.x);
  return (w >> (8 * (k & 3))) & 0xFFu;
}

struct SplitArgs {
  const uint4* text; uint32_t form; uint32_t n_tiles;
  uint32_t* tile_fn; uint32_t* tile_state;     // composed map of each tile; string state at each tile's first byte
  int* tile_dd; long long* tile_depth;         // depth change of each tile; depth before each tile's first byte
  uint32_t* tile_cnt;                          // starts | ends << 16 of each tile
  unsigned long long* tile_off;                // records starting / ending before each tile (2 words per tile)
  unsigned long long* starts; unsigned long long* ends;   // record start positions; one past each record's last byte
  unsigned long long* sum;
};

// PHASE 0: each tile's composed map.  1: each tile's depth change (array form).  2: record starts and ends per tile,
// the closing byte and the last non-blank byte.  3: the positions of the starts and ends.
template <int PHASE>
__global__ void __launch_bounds__(SPLIT_THREADS) inputs_split_kernel(SplitArgs a) {
  const uint32_t tile = blockIdx.x;
  const size_t base = (size_t)tile * SPLIT_TILE + (size_t)threadIdx.x * SPLIT_BYTES;
  uint4 b[SPLIT_BYTES / 16];
#pragma unroll
  for (int k = 0; k < SPLIT_BYTES / 16; k++) b[k] = a.text[base / 16 + k];
  uint32_t f = FN_ID, total_f;
  for (int k = 0; k < SPLIT_BYTES; k++) f = FnThen()(f, byte_fn(a.form, byte_of(b, k)));
  if (PHASE == 0) {
    block_scan(f, FN_ID, FnThen(), &total_f);
    if (threadIdx.x == 0) a.tile_fn[tile] = total_f;
    return;
  }
  uint32_t s = fn_apply(block_scan(f, FN_ID, FnThen(), &total_f), a.tile_state[tile]);
  const uint32_t s0 = s;
  long long depth = 0;
  if (a.form == FORM_ARRAY) {
    int dd = 0;
    for (int k = 0; k < SPLIT_BYTES; k++) {
      const uint32_t c = byte_of(b, k);
      if (s == S_OUT) dd += (c == '[' || c == '{') ? 1 : (c == ']' || c == '}') ? -1 : 0;
      s = fn_apply(byte_fn(a.form, c), s);
    }
    int total_dd;
    const int ex = block_scan(dd, 0, Add(), &total_dd);
    if (PHASE == 1) {
      if (threadIdx.x == 0) a.tile_dd[tile] = total_dd;
      return;
    }
    depth = a.tile_depth[tile] + ex;
    s = s0;
  }
  if (PHASE == 1) return;
  // record starts (low half) and ends (high half) in this thread's bytes
  uint32_t cnt = 0;
  unsigned long long close = ~0ull, last = 0;
  unsigned long long o_start = 0, o_end = 0;
  if (PHASE == 3) {
    uint32_t c2 = 0;
    {
      uint32_t ss = s; long long d = depth;
      for (int k = 0; k < SPLIT_BYTES; k++) {
        const uint32_t c = byte_of(b, k);
        if (a.form == FORM_LINES) c2 += (ss == 0 && !is_ws(c));
        else if (ss == S_OUT) {
          c2 += (c == '{' && d == 1) + ((c == '}' && d == 2) << 16);
          d += (c == '[' || c == '{') ? 1 : (c == ']' || c == '}') ? -1 : 0;
        }
        ss = fn_apply(byte_fn(a.form, c), ss);
      }
    }
    uint32_t tot;
    const uint32_t ex = block_scan(c2, 0u, Add(), &tot);
    o_start = a.tile_off[2 * tile] + (ex & 0xFFFFu);
    o_end = a.tile_off[2 * tile + 1] + (ex >> 16);
  }
  for (int k = 0; k < SPLIT_BYTES; k++) {
    const uint32_t c = byte_of(b, k);
    const unsigned long long pos = base + k;
    if (a.form == FORM_LINES) {
      if (s == 0 && !is_ws(c)) {
        if (PHASE == 3) a.starts[o_start++] = pos;
        cnt++;
      }
    } else {
      if (!is_ws(c)) last = pos + 1;
      if (s == S_OUT) {
        if (c == '{' && depth == 1) { if (PHASE == 3) a.starts[o_start++] = pos; cnt++; }
        if (c == '}' && depth == 2) { if (PHASE == 3) a.ends[o_end++] = pos + 1; cnt += 1u << 16; }
        if ((c == '}' || c == ']') && depth == 1 && close == ~0ull) close = pos;
        depth += (c == '[' || c == '{') ? 1 : (c == ']' || c == '}') ? -1 : 0;
      }
    }
    s = fn_apply(byte_fn(a.form, c), s);
  }
  if (PHASE == 2) {
    uint32_t tot;
    block_scan(cnt, 0u, Add(), &tot);
    if (threadIdx.x == 0) a.tile_cnt[tile] = tot;
    if (a.form == FORM_ARRAY) {
      for (int o = 16; o > 0; o >>= 1) {
        last = max(last, __shfl_down_sync(0xFFFFFFFFu, last, o));
        close = min(close, __shfl_down_sync(0xFFFFFFFFu, close, o));
      }
      if ((threadIdx.x & 31) == 0) {
        if (last) atomicMax(&a.sum[SUM_LAST], last);
        if (close != ~0ull) atomicMin(&a.sum[SUM_CLOSE], close);
      }
    }
  }
}

// scans over the tiles, one block: every thread walks a contiguous run of tiles
__global__ void __launch_bounds__(SCAN_THREADS) inputs_tile_scan_kernel(int what, SplitArgs a) {
  __shared__ unsigned long long part[SCAN_THREADS][2];
  const uint32_t per = (a.n_tiles + SCAN_THREADS - 1) / SCAN_THREADS;
  const uint32_t lo = min(a.n_tiles, threadIdx.x * per), hi = min(a.n_tiles, lo + per);
  unsigned long long x = what == 0 ? FN_ID : 0, y = 0;
  for (uint32_t t = lo; t < hi; t++) {
    if (what == 0) x = FnThen()((uint32_t)x, a.tile_fn[t]);
    else if (what == 1) x += (unsigned long long)(long long)a.tile_dd[t];
    else { x += a.tile_cnt[t] & 0xFFFFu; y += a.tile_cnt[t] >> 16; }
  }
  part[threadIdx.x][0] = x; part[threadIdx.x][1] = y;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long px = what == 0 ? FN_ID : 0, py = 0;
    for (int k = 0; k < SCAN_THREADS; k++) {
      const unsigned long long vx = part[k][0], vy = part[k][1];
      part[k][0] = px; part[k][1] = py;
      if (what == 0) px = FnThen()((uint32_t)px, (uint32_t)vx);
      else { px += vx; py += vy; }
    }
    if (what == 2) { a.sum[SUM_STARTS] = px; a.sum[SUM_ENDS] = py; }
  }
  __syncthreads();
  x = part[threadIdx.x][0]; y = part[threadIdx.x][1];
  for (uint32_t t = lo; t < hi; t++) {
    if (what == 0) { a.tile_state[t] = fn_apply((uint32_t)x, 0); x = FnThen()((uint32_t)x, a.tile_fn[t]); }
    else if (what == 1) { a.tile_depth[t] = (long long)x; x += (unsigned long long)(long long)a.tile_dd[t]; }
    else { a.tile_off[2 * t] = x; a.tile_off[2 * t + 1] = y; x += a.tile_cnt[t] & 0xFFFFu; y += a.tile_cnt[t] >> 16; }
  }
}

// the text of one record, 16 bytes at a time; -1 past the record (and, in JSON Lines, at a newline)
struct Reader {
  const uint4* t; unsigned long long lim; bool lines; unsigned long long cur; uint4 w;
  __device__ int at(unsigned long long p) {
    if (p >= lim) return -1;
    if ((p >> 4) != cur) { cur = p >> 4; w = __ldg(t + cur); }
    const uint32_t x = (p & 8) ? ((p & 4) ? w.w : w.z) : ((p & 4) ? w.y : w.x);
    const int c = (int)((x >> (8 * (p & 3))) & 0xFFu);
    return (lines && c == '\n') ? -1 : c;
  }
  __device__ unsigned long long ws(unsigned long long p) {
    for (int c = at(p); c >= 0 && is_ws((uint32_t)c); c = at(++p)) {}
    return p;
  }
};

struct ParseArgs {
  const uint4* text; unsigned long long len; uint32_t form; uint32_t check_pairs;
  const unsigned long long* starts; const unsigned long long* ends;    // ends: array form only
  size_t n;
  const uint4* slots; uint32_t slot_mask;      // key hash table: {hash, name offset, name length, key + 1 (0: empty)}
  const uint4* keys; const uint8_t* names;     // per key: {signal offset, length, fits the row}
  uint32_t seen_words; uint32_t* seen;         // per record: which keys it has named
  uint4* rows; uint32_t I;
  unsigned long long* marks;                   // per marked record: index, start, end
  unsigned long long* sum;
};

__device__ __forceinline__ uint32_t fnv1a(uint32_t h, uint32_t c) { return (h ^ c) * 16777619u; }

// r = r * scale + add on 8 little-endian 32-bit limbs; false when the result does not fit 256 bits
__device__ __forceinline__ bool mul_add(uint32_t* r, uint32_t scale, uint32_t add) {
  unsigned long long c = add;
#pragma unroll
  for (int i = 0; i < 8; i++) { c += (unsigned long long)r[i] * scale; r[i] = (uint32_t)c; c >>= 32; }
  return c == 0;
}

// one value at p: "<decimal digits>" or a bare integer that fits u64.  Returns the position after it, or ~0 when the
// record has to go to the host
__device__ unsigned long long parse_scalar(Reader& rd, unsigned long long p, uint32_t* v) {
#pragma unroll
  for (int i = 0; i < 8; i++) v[i] = 0;
  int c = rd.at(p);
  if (c == '"') {
    uint32_t chunk = 0, scale = 1, nd = 0;
    for (c = rd.at(++p); c >= '0' && c <= '9'; c = rd.at(++p)) {
      chunk = chunk * 10 + (uint32_t)(c - '0'); scale *= 10; nd++;
      if (scale == 1000000000u) { if (!mul_add(v, scale, chunk)) return ~0ull; chunk = 0; scale = 1; }
    }
    if (c != '"' || nd == 0) return ~0ull;       // escapes, underscores, other bytes, "": the host decides
    if (scale > 1 && !mul_add(v, scale, chunk)) return ~0ull;
    return p + 1;
  }
  if (c >= '0' && c <= '9') {
    unsigned long long x = 0;
    for (; c >= '0' && c <= '9'; c = rd.at(++p)) {
      const unsigned long long d = (unsigned long long)(c - '0');
      if (x > (~0ull - d) / 10) return ~0ull;      // the host's u64 rule (inputs.cpp: J::number)
      x = x * 10 + d;
    }
    if (c == '.' || c == 'e' || c == 'E') return ~0ull;
    v[0] = (uint32_t)x; v[1] = (uint32_t)(x >> 32);
    return p;
  }
  return ~0ull;
}

__global__ void __launch_bounds__(PARSE_THREADS) inputs_parse_kernel(ParseArgs a) {
  const size_t r = (size_t)blockIdx.x * PARSE_THREADS + threadIdx.x;
  if (r >= a.n) return;
  const unsigned long long start = a.starts[r];
  Reader rd{a.text, a.form == FORM_LINES ? a.len : a.ends[r], a.form == FORM_LINES, ~0ull, make_uint4(0, 0, 0, 0)};
  if (a.check_pairs && !(start < a.ends[r] && (r + 1 == a.n || a.ends[r] <= a.starts[r + 1]))) {
    atomicOr((unsigned int*)&a.sum[SUM_ODD], 1u);   // not the host's pairing of starts and ends: the host splits
    return;
  }
  uint4* row = a.rows + r * (size_t)a.I * 2;
  uint32_t* seen = a.seen + r * (size_t)a.seen_words;
  for (uint32_t k = 0; k < a.seen_words; k++) seen[k] = 0;
  for (uint32_t k = 0; k < a.I; k++) { row[2 * k] = make_uint4(k == 0, 0, 0, 0); row[2 * k + 1] = make_uint4(0, 0, 0, 0); }
  bool ok = a.I > 0;
  unsigned long long p = rd.ws(start);
  if (ok && rd.at(p) == '{') {
    p = rd.ws(p + 1);
    if (rd.at(p) == '}') p++;
    else while (true) {
      // key
      if (rd.at(p) != '"') { ok = false; break; }
      const unsigned long long k0 = ++p;
      uint32_t h = 2166136261u;
      int c;
      for (c = rd.at(p); c >= 0 && c != '"' && c != '\\'; c = rd.at(++p)) h = fnv1a(h, (uint32_t)c);
      if (c != '"') { ok = false; break; }
      const uint32_t klen = (uint32_t)(p - k0);
      uint32_t key = 0;
      for (uint32_t i = h & a.slot_mask;; i = (i + 1) & a.slot_mask) {
        const uint4 e = __ldg(a.slots + i);
        if (e.w == 0) break;
        if (e.x != h || e.z != klen) continue;
        uint32_t j = 0;
        while (j < klen && a.names[e.y + j] == (uint8_t)rd.at(k0 + j)) j++;
        if (j == klen) { key = e.w; break; }
      }
      if (key == 0) { ok = false; break; }           // unknown signal
      key--;
      if (seen[key >> 5] & (1u << (key & 31))) { ok = false; break; }   // repeated: the last value would win
      seen[key >> 5] |= 1u << (key & 31);
      const uint4 info = __ldg(a.keys + key);
      if (!info.z) { ok = false; break; }            // the signal does not fit the row
      p = rd.ws(p + 1);
      if (rd.at(p) != ':') { ok = false; break; }
      p = rd.ws(p + 1);
      uint32_t n_vals = 0, v[8];
      if (rd.at(p) == '[') {
        p = rd.ws(p + 1);
        if (rd.at(p) == ']') p++;
        else while (true) {
          p = parse_scalar(rd, p, v);
          if (p == ~0ull || n_vals >= info.y) { ok = false; break; }
          uint4* dst = row + 2 * (size_t)(info.x + n_vals);
          dst[0] = make_uint4(v[0], v[1], v[2], v[3]); dst[1] = make_uint4(v[4], v[5], v[6], v[7]);
          n_vals++;
          p = rd.ws(p);
          c = rd.at(p);
          if (c == ',') { p = rd.ws(p + 1); continue; }
          if (c == ']') { p++; break; }
          ok = false; break;
        }
        if (!ok) break;
      } else {
        p = parse_scalar(rd, p, v);
        if (p == ~0ull || info.y < 1) { ok = false; break; }
        uint4* dst = row + 2 * (size_t)info.x;
        dst[0] = make_uint4(v[0], v[1], v[2], v[3]); dst[1] = make_uint4(v[4], v[5], v[6], v[7]);
        n_vals = 1;
      }
      if (n_vals != info.y) { ok = false; break; }
      p = rd.ws(p);
      c = rd.at(p);
      if (c == ',') { p = rd.ws(p + 1); continue; }
      if (c == '}') { p++; break; }
      ok = false; break;
    }
    if (ok) ok = rd.at(rd.ws(p)) < 0;                // nothing but blanks after the object
  } else ok = false;
  if (ok) return;
  // marked: the host parses this record from its text
  unsigned long long end = rd.lim;
  if (a.form == FORM_LINES) {
    if (p == ~0ull) p = start;
    while (rd.at(p) >= 0) p++;                       // the newline or the end of the text
    rd.lines = false;
    while (p > start && is_blank((uint32_t)rd.at(p - 1))) p--;
    end = p;
  }
  const unsigned long long m = atomicAdd(&a.sum[SUM_MARKS], 1ull);
  a.marks[3 * m] = r; a.marks[3 * m + 1] = start; a.marks[3 * m + 2] = end;
}

// rows parsed by the host -> their places among the device rows
__global__ void inputs_scatter_kernel(const uint4* src, const uint32_t* idx, uint32_t n_rows, uint32_t row_quads, uint4* rows) {
  for (uint32_t j = blockIdx.x; j < n_rows; j += gridDim.x)
    for (uint32_t k = threadIdx.x; k < row_quads; k += blockDim.x) rows[(size_t)idx[j] * row_quads + k] = src[(size_t)j * row_quads + k];
}

template <typename T> void grow(T*& p, size_t& cap, size_t n) {
  if (n <= cap) return;
  cudaFree(p); p = nullptr; cap = 0;
  CUDA_CHECK(cudaMalloc(&p, n * sizeof(T)));
  cap = n;
}

}  // namespace

// per device: the key table of the graph and scratch that grows with the largest text seen
struct DeviceInputs::Dev {
  int device = -1;
  std::mutex mu;                               // one call at a time per graph and device
  uint4* slots = nullptr; uint4* keys = nullptr; uint8_t* names = nullptr;
  uint32_t slot_mask = 0, n_keys = 0;
  uint4* text = nullptr; size_t text_cap = 0;
  uint32_t* tile_fn = nullptr; size_t tile_fn_cap = 0;
  uint32_t* tile_state = nullptr; size_t tile_state_cap = 0;
  int* tile_dd = nullptr; size_t tile_dd_cap = 0;
  long long* tile_depth = nullptr; size_t tile_depth_cap = 0;
  uint32_t* tile_cnt = nullptr; size_t tile_cnt_cap = 0;
  unsigned long long* tile_off = nullptr; size_t tile_off_cap = 0;
  unsigned long long* starts = nullptr; size_t starts_cap = 0;
  unsigned long long* ends = nullptr; size_t ends_cap = 0;
  uint32_t* seen = nullptr; size_t seen_cap = 0;
  unsigned long long* marks = nullptr; size_t marks_cap = 0;
  unsigned long long* sum = nullptr;
  unsigned long long* h_sum = nullptr;         // pinned
  ~Dev() {
    int prev = -1;
    cudaGetDevice(&prev);
    cudaSetDevice(device);
    cudaFree(slots); cudaFree(keys); cudaFree(names); cudaFree(text);
    cudaFree(tile_fn); cudaFree(tile_state); cudaFree(tile_dd); cudaFree(tile_depth); cudaFree(tile_cnt); cudaFree(tile_off);
    cudaFree(starts); cudaFree(ends); cudaFree(seen); cudaFree(marks); cudaFree(sum);
    cudaFreeHost(h_sum);
    if (prev >= 0) cudaSetDevice(prev);
  }
};

DeviceInputs::DeviceInputs(const Graph& g) : g(g) {}
DeviceInputs::~DeviceInputs() = default;

DeviceInputs::Dev* DeviceInputs::dev(int device) {
  std::lock_guard<std::mutex> lk(mu);
  auto it = devs.find(device);
  if (it != devs.end()) return it->second.get();
  check_device(device);
  DeviceGuard on(device);
  std::unique_ptr<Dev> d(new Dev());
  d->device = device;
  // the key table: open addressing on the FNV-1a hash of the name, at most half full
  std::vector<uint4> keys;
  std::vector<uint8_t> names;
  std::vector<std::pair<uint32_t, uint32_t>> at;   // hash, name offset
  for (auto& kv : g.inputs) {
    const uint32_t off = kv.second.first, ln = kv.second.second;
    uint32_t h = 2166136261u;
    for (unsigned char c : kv.first) h = (h ^ c) * 16777619u;
    at.emplace_back(h, (uint32_t)names.size());
    names.insert(names.end(), kv.first.begin(), kv.first.end());
    keys.push_back(make_uint4(off, ln, (size_t)off + ln <= g.inputs_size ? 1u : 0u, 0));
  }
  size_t n_slots = 2;
  while (n_slots < 2 * keys.size()) n_slots *= 2;
  std::vector<uint4> slots(n_slots, make_uint4(0, 0, 0, 0));
  size_t k = 0;
  for (auto& kv : g.inputs) {
    size_t i = at[k].first & (n_slots - 1);
    while (slots[i].w) i = (i + 1) & (n_slots - 1);
    slots[i] = make_uint4(at[k].first, at[k].second, (uint32_t)kv.first.size(), (uint32_t)k + 1);
    k++;
  }
  d->slot_mask = (uint32_t)(n_slots - 1);
  d->n_keys = (uint32_t)keys.size();
  CUDA_CHECK(cudaMalloc(&d->slots, n_slots * sizeof(uint4)));
  CUDA_CHECK(cudaMemcpy(d->slots, slots.data(), n_slots * sizeof(uint4), cudaMemcpyHostToDevice));
  CUDA_CHECK(cudaMalloc(&d->keys, std::max<size_t>(keys.size(), 1) * sizeof(uint4)));
  CUDA_CHECK(cudaMemcpy(d->keys, keys.data(), keys.size() * sizeof(uint4), cudaMemcpyHostToDevice));
  CUDA_CHECK(cudaMalloc(&d->names, std::max<size_t>(names.size(), 1)));
  CUDA_CHECK(cudaMemcpy(d->names, names.data(), names.size(), cudaMemcpyHostToDevice));
  CUDA_CHECK(cudaMalloc(&d->sum, SUM_WORDS * 8));
  CUDA_CHECK(cudaHostAlloc(&d->h_sum, SUM_WORDS * 8, cudaHostAllocDefault));
  return (devs[device] = std::move(d)).get();
}

void DeviceInputs::parse(int device, const char* text, size_t len, void* d_rows, size_t max_sets, void* stream, size_t* n_sets) {
  *n_sets = 0;
  Dev* d = dev(device);
  DeviceGuard on(device);
  std::lock_guard<std::mutex> lk(d->mu);
  cudaStream_t s = (cudaStream_t)stream;
  // the form is that of the first non-blank byte (split_records)
  size_t i0 = 0;
  while (i0 < len && (text[i0] == ' ' || text[i0] == '\t' || text[i0] == '\n' || text[i0] == '\r')) i0++;
  const uint32_t form = (i0 < len && text[i0] == '[') ? FORM_ARRAY : FORM_LINES;
  const size_t n_tiles = (len + SPLIT_TILE - 1) / SPLIT_TILE;
  if (n_tiles > 0xFFFFFFFFull) throw Error("input text too large");
  if (n_tiles == 0) return;                      // no text, no record
  grow(d->text, d->text_cap, n_tiles * SPLIT_TILE / 16);
  CUDA_CHECK(cudaMemcpyAsync(d->text, text, len, cudaMemcpyHostToDevice, s));
  CUDA_CHECK(cudaMemsetAsync((char*)d->text + len, ' ', n_tiles * SPLIT_TILE - len, s));   // padding: blanks
  grow(d->tile_fn, d->tile_fn_cap, n_tiles); grow(d->tile_state, d->tile_state_cap, n_tiles);
  grow(d->tile_cnt, d->tile_cnt_cap, n_tiles); grow(d->tile_off, d->tile_off_cap, 2 * n_tiles);
  if (form == FORM_ARRAY) { grow(d->tile_dd, d->tile_dd_cap, n_tiles); grow(d->tile_depth, d->tile_depth_cap, n_tiles); }
  CUDA_CHECK(cudaMemsetAsync(d->sum, 0, SUM_WORDS * 8, s));
  CUDA_CHECK(cudaMemsetAsync(d->sum + SUM_CLOSE, 0xFF, 8, s));
  SplitArgs a;
  a.text = d->text; a.form = form; a.n_tiles = (uint32_t)n_tiles;
  a.tile_fn = d->tile_fn; a.tile_state = d->tile_state; a.tile_dd = d->tile_dd; a.tile_depth = d->tile_depth;
  a.tile_cnt = d->tile_cnt; a.tile_off = d->tile_off; a.starts = nullptr; a.ends = nullptr; a.sum = d->sum;
  const unsigned grid = (unsigned)n_tiles;
  inputs_split_kernel<0><<<grid, SPLIT_THREADS, 0, s>>>(a);
  inputs_tile_scan_kernel<<<1, SCAN_THREADS, 0, s>>>(0, a);
  if (form == FORM_ARRAY) {
    inputs_split_kernel<1><<<grid, SPLIT_THREADS, 0, s>>>(a);
    inputs_tile_scan_kernel<<<1, SCAN_THREADS, 0, s>>>(1, a);
  }
  inputs_split_kernel<2><<<grid, SPLIT_THREADS, 0, s>>>(a);
  inputs_tile_scan_kernel<<<1, SCAN_THREADS, 0, s>>>(2, a);
  CUDA_CHECK(cudaGetLastError());
  CUDA_CHECK(cudaMemcpyAsync(d->h_sum, d->sum, SUM_WORDS * 8, cudaMemcpyDeviceToHost, s));
  CUDA_CHECK(cudaStreamSynchronize(s));
  const unsigned long long n_starts = d->h_sum[SUM_STARTS], n_ends = d->h_sum[SUM_ENDS];
  std::vector<std::pair<size_t, size_t>> host_rec;
  bool host_split = false;
  if (form == FORM_ARRAY) {
    // an unterminated array or bytes after it: split_records throws the host's message
    if (d->h_sum[SUM_CLOSE] == ~0ull || d->h_sum[SUM_LAST] > d->h_sum[SUM_CLOSE] + 1) {
      split_records(text, len, host_rec);
      host_split = true;
    } else if (n_starts != n_ends) {             // an element that is not an object at depth 1: the host pairs them
      split_records(text, len, host_rec);
      host_split = true;
    }
  }
  const size_t n = host_split ? host_rec.size() : (size_t)(form == FORM_LINES ? n_starts : n_ends);
  *n_sets = n;
  if (n > max_sets)
    throw Error("the text holds " + std::to_string(n) + " input sets, more than max_sets = " + std::to_string(max_sets));
  if (n == 0) return;
  if (n > 0xFFFFFFFFull) throw Error("more than 2^32 - 1 input sets in one text");
  const uint32_t seen_words = (d->n_keys + 31) / 32;
  grow(d->starts, d->starts_cap, n); grow(d->marks, d->marks_cap, 3 * n);
  grow(d->seen, d->seen_cap, std::max<size_t>(n * seen_words, 1));
  if (form == FORM_ARRAY) grow(d->ends, d->ends_cap, n);
  auto upload_host_split = [&]() {
    std::vector<unsigned long long> st(n), en(n);
    for (size_t r = 0; r < n; r++) { st[r] = host_rec[r].first; en[r] = host_rec[r].second; }
    CUDA_CHECK(cudaMemcpyAsync(d->starts, st.data(), n * 8, cudaMemcpyHostToDevice, s));
    CUDA_CHECK(cudaMemcpyAsync(d->ends, en.data(), n * 8, cudaMemcpyHostToDevice, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
  };
  if (host_split) upload_host_split();
  else {
    a.starts = d->starts; a.ends = d->ends;
    inputs_split_kernel<3><<<grid, SPLIT_THREADS, 0, s>>>(a);
    CUDA_CHECK(cudaGetLastError());
  }
  ParseArgs pa;
  pa.text = d->text; pa.len = len; pa.form = form; pa.check_pairs = form == FORM_ARRAY && !host_split;
  pa.starts = d->starts; pa.ends = d->ends; pa.n = n;
  pa.slots = d->slots; pa.slot_mask = d->slot_mask; pa.keys = d->keys; pa.names = d->names;
  pa.seen_words = seen_words; pa.seen = d->seen;
  pa.rows = (uint4*)d_rows; pa.I = g.inputs_size; pa.marks = d->marks; pa.sum = d->sum;
  const unsigned pgrid = (unsigned)((n + PARSE_THREADS - 1) / PARSE_THREADS);
  inputs_parse_kernel<<<pgrid, PARSE_THREADS, 0, s>>>(pa);
  CUDA_CHECK(cudaGetLastError());
  CUDA_CHECK(cudaMemcpyAsync(d->h_sum, d->sum, SUM_WORDS * 8, cudaMemcpyDeviceToHost, s));
  CUDA_CHECK(cudaStreamSynchronize(s));
  const bool odd = d->h_sum[SUM_ODD] != 0;
  if (odd) {
    // starts and ends do not pair up one to one (a depth-1 element that is not an object): the host's split decides
    split_records(text, len, host_rec);
    upload_host_split();
    pa.check_pairs = 0;
    CUDA_CHECK(cudaMemsetAsync(d->sum, 0, SUM_WORDS * 8, s));
    inputs_parse_kernel<<<pgrid, PARSE_THREADS, 0, s>>>(pa);
    CUDA_CHECK(cudaGetLastError());
    CUDA_CHECK(cudaMemcpyAsync(d->h_sum, d->sum, SUM_WORDS * 8, cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
  }
  const size_t n_marks = (size_t)d->h_sum[SUM_MARKS];
  // GW_TRACE_HOST=1: how the text was split and how many records the host had to parse
  const char* trace = getenv("GW_TRACE_HOST");
  if (trace && atoi(trace) != 0)
    fprintf(stderr, "[gw inputs] form %s, records %zu, host split %d, marked %zu\n", form == FORM_ARRAY ? "array" : "lines", n,
            host_split || odd ? 1 : 0, n_marks);
  if (n_marks == 0) return;
  // the marked records, in record order: the first that fails is the lowest failing record of the text
  std::vector<unsigned long long> mk(3 * n_marks);
  CUDA_CHECK(cudaMemcpyAsync(mk.data(), d->marks, mk.size() * 8, cudaMemcpyDeviceToHost, s));
  CUDA_CHECK(cudaStreamSynchronize(s));
  std::vector<size_t> order(n_marks);
  for (size_t j = 0; j < n_marks; j++) order[j] = j;
  std::sort(order.begin(), order.end(), [&](size_t x, size_t y) { return mk[3 * x] < mk[3 * y]; });
  const size_t I = g.inputs_size;
  std::vector<U256> host_rows(n_marks * I);
  std::vector<uint32_t> idx(n_marks);
  for (size_t j = 0; j < n_marks; j++) {
    const unsigned long long* m = &mk[3 * order[j]];
    idx[j] = (uint32_t)m[0];
    try {
      std::vector<U256> row = build_inputs_buffer(g, deserialize_inputs(text + m[1], (size_t)(m[2] - m[1])));
      std::copy(row.begin(), row.end(), host_rows.begin() + j * I);
    } catch (const std::exception& e) {
      throw Error("input set " + std::to_string(m[0] + 1) + ": " + e.what());
    }
  }
  uint4* src = nullptr; uint32_t* d_idx = nullptr;
  CUDA_CHECK(cudaMallocAsync(&src, host_rows.size() * 32, s));
  CUDA_CHECK(cudaMallocAsync(&d_idx, n_marks * 4, s));
  CUDA_CHECK(cudaMemcpyAsync(src, host_rows.data(), host_rows.size() * 32, cudaMemcpyHostToDevice, s));
  CUDA_CHECK(cudaMemcpyAsync(d_idx, idx.data(), n_marks * 4, cudaMemcpyHostToDevice, s));
  inputs_scatter_kernel<<<(unsigned)std::min<size_t>(n_marks, 4096), 128, 0, s>>>(src, d_idx, (uint32_t)n_marks, (uint32_t)(I * 2), (uint4*)d_rows);
  CUDA_CHECK(cudaGetLastError());
  CUDA_CHECK(cudaFreeAsync(src, s));
  CUDA_CHECK(cudaFreeAsync(d_idx, s));
  CUDA_CHECK(cudaStreamSynchronize(s));
}

}  // namespace gw
