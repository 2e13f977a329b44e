#include "inputs.hpp"

#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <mutex>
#include <thread>

namespace gw {

namespace {
struct J {
  const char* p; const char* end;
  void ws() { while (p < end && (*p == ' ' || *p == '\t' || *p == '\n' || *p == '\r')) p++; }
  [[noreturn]] void fail(const char* what) { throw Error(std::string("Failed to parse inputs: invalid JSON: ") + what); }
  char peek() { ws(); if (p >= end) fail("unexpected end"); return *p; }
  void expect(char c) { if (peek() != c) fail("unexpected character"); p++; }
  std::string str() {
    expect('"');
    std::string s;
    while (true) {
      if (p >= end) fail("unterminated string");
      char c = *p++;
      if (c == '"') break;
      if (c == '\\') {
        if (p >= end) fail("bad escape");
        char e = *p++;
        switch (e) {
          case '"': s += '"'; break; case '\\': s += '\\'; break; case '/': s += '/'; break;
          case 'b': s += '\b'; break; case 'f': s += '\f'; break; case 'n': s += '\n'; break;
          case 'r': s += '\r'; break; case 't': s += '\t'; break;
          case 'u': {
            if (end - p < 4) fail("bad \\u escape");
            unsigned cp = 0;
            for (int i = 0; i < 4; i++) {
              char h = *p++; cp <<= 4;
              if (h >= '0' && h <= '9') cp |= h - '0'; else if (h >= 'a' && h <= 'f') cp |= h - 'a' + 10;
              else if (h >= 'A' && h <= 'F') cp |= h - 'A' + 10; else fail("bad \\u escape");
            }
            if (cp < 0x80) s += (char)cp;
            else if (cp < 0x800) { s += (char)(0xC0 | (cp >> 6)); s += (char)(0x80 | (cp & 0x3F)); }
            else { s += (char)(0xE0 | (cp >> 12)); s += (char)(0x80 | ((cp >> 6) & 0x3F)); s += (char)(0x80 | (cp & 0x3F)); }
            break;
          }
          default: fail("bad escape");
        }
      } else s += c;
    }
    return s;
  }
  // a JSON number; accepted as a value only if it is a non-negative integer that fits u64 (lib.rs:211-214)
  bool number(uint64_t* out) {
    ws();
    const char* s = p;
    bool neg = false, integral = true;
    if (p < end && *p == '-') { neg = true; p++; }
    if (p >= end || *p < '0' || *p > '9') fail("bad number");
    while (p < end && *p >= '0' && *p <= '9') p++;
    if (p < end && *p == '.') { integral = false; p++; while (p < end && *p >= '0' && *p <= '9') p++; }
    if (p < end && (*p == 'e' || *p == 'E')) { integral = false; p++; if (p < end && (*p == '+' || *p == '-')) p++; while (p < end && *p >= '0' && *p <= '9') p++; }
    if (neg || !integral) return false;
    uint64_t v = 0;
    for (const char* q = s; q < p; q++) {
      uint64_t d = (uint64_t)(*q - '0');
      if (v > (UINT64_MAX - d) / 10) return false;
      v = v * 10 + d;
    }
    *out = v;
    return true;
  }
  void skip_value() {   // only used to give a precise error for unsupported value kinds
    char c = peek();
    if (c == '{') { p++; if (peek() == '}') { p++; return; } while (true) { str(); expect(':'); skip_value(); if (peek() == ',') { p++; continue; } expect('}'); return; } }
    if (c == '[') { p++; if (peek() == ']') { p++; return; } while (true) { skip_value(); if (peek() == ',') { p++; continue; } expect(']'); return; } }
    if (c == '"') { str(); return; }
    if (c == 't' && end - p >= 4 && !memcmp(p, "true", 4)) { p += 4; return; }
    if (c == 'f' && end - p >= 5 && !memcmp(p, "false", 5)) { p += 5; return; }
    if (c == 'n' && end - p >= 4 && !memcmp(p, "null", 4)) { p += 4; return; }
    uint64_t v; number(&v);
  }
};

U256 parse_scalar(J& j, const std::string& key, bool in_array) {
  char c = j.peek();
  if (c == '"') {
    // the common case, without a std::string: "<decimal digits>"
    const char* q = j.p + 1;
    while (q < j.end && *q >= '0' && *q <= '9') q++;
    U256 fast;
    if (q < j.end && *q == '"' && q > j.p + 1 && u256_parse_dec_digits(j.p + 1, (size_t)(q - j.p - 1), &fast)) { j.p = q + 1; return fast; }
    std::string s = j.str();
    U256 v;
    if (!u256_parse_dec(s, &v)) throw Error("Failed to calculate witness: InputFieldNumberParseError(\"" + s + "\")");
    return v;
  }
  if (c == '-' || (c >= '0' && c <= '9')) {
    uint64_t v;
    if (!j.number(&v)) throw Error("Failed to calculate witness: InputsUnmarshal(\"signal value is not a positive integer\")");
    return u256_from_u64(v);
  }
  if (in_array) throw Error("Failed to calculate witness: InputsUnmarshal(\"inputs must be a string: " + key + "\")");
  throw Error("Failed to calculate witness: InputsUnmarshal(\"value for key " + key +
              " must be an a number as a string, as a number of an array of strings of numbers\")");
}
}  // namespace

InputList deserialize_inputs(const char* json, size_t len) {
  J j{json, json + len};
  if (j.peek() != '{') {
    j.skip_value();
    throw Error("Failed to calculate witness: InputsUnmarshal(\"inputs must be an object\")");
  }
  j.p++;
  InputList out;
  if (j.peek() == '}') { j.p++; }
  else {
    while (true) {
      std::string key = j.str();
      j.expect(':');
      std::vector<U256> vals;
      if (j.peek() == '[') {
        j.p++;
        if (j.peek() == ']') j.p++;
        else while (true) {
          vals.push_back(parse_scalar(j, key, true));
          if (j.peek() == ',') { j.p++; continue; }
          j.expect(']');
          break;
        }
      } else vals.push_back(parse_scalar(j, key, false));
      // serde_json::Map keeps the last value of a duplicated key
      bool replaced = false;
      for (auto& kv : out) if (kv.first == key) { kv.second = vals; replaced = true; }
      if (!replaced) out.emplace_back(key, std::move(vals));
      if (j.peek() == ',') { j.p++; continue; }
      j.expect('}');
      break;
    }
  }
  j.ws();
  if (j.p != j.end) j.fail("trailing characters");
  return out;
}

std::vector<U256> build_inputs_buffer(const Graph& g, const InputList& inputs) {
  if (g.inputs_size == 0) throw Error("Failed to calculate witness: graph without an input buffer");
  std::vector<U256> buf(g.inputs_size, u256_from_u64(0));
  buf[0] = u256_from_u64(1);
  for (auto& kv : inputs) {
    auto it = g.inputs.find(kv.first);
    if (it == g.inputs.end()) throw Error("Failed to calculate witness: unknown input signal " + kv.first);
    uint32_t off = it->second.first, ln = it->second.second;
    if (ln != kv.second.size()) throw Error("Failed to calculate witness: Invalid input length for " + kv.first);
    if ((size_t)off + ln > buf.size()) throw Error("Failed to calculate witness: input " + kv.first + " out of range");
    for (uint32_t i = 0; i < ln; i++) buf[off + i] = kv.second[i];
  }
  return buf;
}


// record boundaries: JSON Lines, or the elements of one top-level array (split at depth-1 commas, strings skipped)
void split_records(const char* text, size_t len, std::vector<std::pair<size_t, size_t>>& rec) {
  size_t i = 0;
  while (i < len && (text[i] == ' ' || text[i] == '\t' || text[i] == '\n' || text[i] == '\r')) i++;
  if (i < len && text[i] == '[') {
    int depth = 0; bool in_str = false; size_t start = 0;
    for (; i < len; i++) {
      const char c = text[i];
      if (in_str) { if (c == '\\') i++; else if (c == '"') in_str = false; continue; }
      if (c == '"') in_str = true;
      else if (c == '[' || c == '{') { if (depth == 1 && c == '{') start = i; depth++; }
      else if (c == ']' || c == '}') {
        depth--;
        if (depth == 1 && c == '}') rec.emplace_back(start, i + 1);
        if (depth == 0) { i++; break; }
      }
    }
    if (depth != 0 || in_str) throw Error("Failed to parse inputs: invalid JSON: unterminated array of input sets");
    for (; i < len; i++) if (!(text[i] == ' ' || text[i] == '\t' || text[i] == '\n' || text[i] == '\r')) throw Error("Failed to parse inputs: invalid JSON: trailing characters");
    return;
  }
  // JSON Lines: memchr finds the line ends (this scan is the serial part of the batch parser)
  size_t ls = 0;
  while (ls <= len) {
    const char* nl = ls < len ? (const char*)memchr(text + ls, '\n', len - ls) : nullptr;
    const size_t k = nl ? (size_t)(nl - text) : len;
    size_t a = ls, b = k;
    while (a < b && (text[a] == ' ' || text[a] == '\t' || text[a] == '\r')) a++;
    while (b > a && (text[b - 1] == ' ' || text[b - 1] == '\t' || text[b - 1] == '\r')) b--;
    if (b > a) rec.emplace_back(a, b);
    ls = k + 1;
  }
}

size_t parse_inputs_batch(const Graph& g, const char* text, size_t len, int n_threads, U256** out_rows) {
  std::vector<std::pair<size_t, size_t>> rec;
  split_records(text, len, rec);
  const size_t n = rec.size(), I = g.inputs_size;
  // every row is written whole by the thread that parses its record: no zero fill, no second copy
  U256* out = (U256*)malloc(std::max<size_t>(n * I * sizeof(U256), 1));
  if (!out) throw Error("Failed to allocate memory for the input buffer");
  *out_rows = out;
  if (n == 0) return 0;
  if (n_threads <= 0) n_threads = (int)std::max(1u, std::thread::hardware_concurrency());
  n_threads = (int)std::min<size_t>((size_t)n_threads, (n + 63) / 64);
  std::atomic<size_t> next(0);
  std::mutex emu; size_t err_rec = (size_t)-1; std::string err;
  auto work = [&]() {
    while (true) {
      const size_t lo = next.fetch_add(64);
      if (lo >= n) break;
      for (size_t r = lo; r < std::min(n, lo + 64); r++) {
        try {
          InputList in = deserialize_inputs(text + rec[r].first, rec[r].second - rec[r].first);
          std::vector<U256> row = build_inputs_buffer(g, in);
          memcpy(&out[r * I], row.data(), I * sizeof(U256));
        } catch (const std::exception& e) {
          std::lock_guard<std::mutex> lk(emu);
          if (r < err_rec) { err_rec = r; err = e.what(); }
        }
      }
    }
  };
  std::vector<std::thread> th;
  for (int t = 1; t < n_threads; t++) th.emplace_back(work);
  work();
  for (auto& t : th) t.join();
  if (err_rec != (size_t)-1) { free(out); *out_rows = nullptr; throw Error("input set " + std::to_string(err_rec + 1) + ": " + err); }
  return n;
}

}  // namespace gw
