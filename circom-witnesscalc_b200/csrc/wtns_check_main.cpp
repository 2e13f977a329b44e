// wtns-check [--all] <circuit.r1cs> <witness.wtns> [more.wtns ...]
// Drop-in for `snarkjs wtns check circuit.r1cs witness.wtns`: checks that each witness satisfies the circuit's
// constraints.  The .wtns headers are checked on the host (version 2, n8 = 32, BN254's prime, one value per wire);
// the payloads of all files are checked on the GPU in one gw_r1cs_check_batch call.  Prints one line per file
// ("OK" or "constraint k not satisfied") and exits 0 only if every file passes.
// --all: the payloads go through one gw_r1cs_abc_batch call instead (plain layout, with the verdicts), and every failing
// file gets one more line per violated constraint, "  constraint k: a * b != c" (decimal values of <A_k,w>, <B_k,w>,
// <C_k,w>, with witness values reduced mod M), then one line per wire that holds a value >= M.
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/graph_witness.h"
#include "r1cs_eval.cuh"

static bool read_file(const char* path, std::vector<uint8_t>& out) {
  FILE* f = fopen(path, "rb");
  if (!f) return false;
  fseek(f, 0, SEEK_END); long n = ftell(f); fseek(f, 0, SEEK_SET);
  if (n < 0) { fclose(f); return false; }
  out.resize((size_t)n);
  size_t got = n ? fread(out.data(), 1, (size_t)n, f) : 0;
  fclose(f);
  return got == (size_t)n;
}

template <class T> static bool get(const std::vector<uint8_t>& b, size_t& pos, T* v) {
  if (pos > b.size() || b.size() - pos < sizeof(T)) return false;
  memcpy(v, b.data() + pos, sizeof(T)); pos += sizeof(T); return true;
}

// the payload offset of a .wtns v2 file with n_wires values: an empty string on success, else the reason it is
// rejected.  Sections may come in any order.
static std::string parse_wtns(const std::vector<uint8_t>& b, uint32_t n_wires, size_t* payload) {
  uint8_t ref[76];
  gw_wtns_header(0, ref);                          // bytes 28..59: BN254's prime as the library writes it
  size_t pos = 0; uint32_t version = 0, n_sections = 0;
  if (b.size() < 4 || memcmp(b.data(), "wtns", 4) != 0) return "not a .wtns file";
  pos = 4;
  if (!get(b, pos, &version) || version != 2) return "unsupported .wtns version (expected 2)";
  if (!get(b, pos, &n_sections)) return "truncated header";
  size_t hdr_pos = 0, hdr_size = 0, wit_size = 0;
  bool have1 = false, have2 = false;
  for (uint32_t s = 0; s < n_sections; s++) {
    uint32_t type = 0; uint64_t size = 0;
    if (!get(b, pos, &type) || !get(b, pos, &size) || size > b.size() - pos) return "truncated file";
    if (type == 1 || type == 2) {
      if (type == 1 ? have1 : have2) return "section " + std::to_string(type) + " appears twice";
      if (type == 1) { have1 = true; hdr_pos = pos; hdr_size = (size_t)size; }
      else { have2 = true; *payload = pos; wit_size = (size_t)size; }
    }
    pos += (size_t)size;
  }
  if (!have1) return "header section (1) missing";
  if (!have2) return "witness section (2) missing";
  uint32_t n8 = 0, n_witness = 0;
  size_t p = hdr_pos;
  if (hdr_size != 40 || !get(b, p, &n8)) return "malformed header section";
  if (n8 != 32) return "field element size is not 32 bytes";
  if (memcmp(b.data() + p, ref + 28, 32) != 0) return "the prime is not BN254's";
  p += 32;
  get(b, p, &n_witness);
  if (wit_size != 32ull * n_witness) return "witness section length does not match the header";
  if (n_witness != n_wires) return "the witness has " + std::to_string(n_witness) + " values, the circuit " + std::to_string(n_wires) + " wires";
  return "";
}

static std::string decimal(const uint8_t* v32) {
  uint32_t l[8];
  memcpy(l, v32, 32);
  std::string s;
  do {
    uint64_t rem = 0;
    for (int i = 7; i >= 0; i--) {
      const uint64_t cur = (rem << 32) | l[i];
      l[i] = (uint32_t)(cur / 10);
      rem = cur % 10;
    }
    s.push_back((char)('0' + rem));
  } while (std::any_of(l, l + 8, [](uint32_t x) { return x != 0; }));
  std::reverse(s.begin(), s.end());
  return s;
}

static gw::fe to_fe(const uint8_t* v32) { gw::fe r; memcpy(r.l, v32, 32); return r; }

int main(int argc, char** argv) {
  const char* prog = argv[0];
  const bool all = argc > 1 && strcmp(argv[1], "--all") == 0;
  if (all) { argv++; argc--; }
  if (argc < 3) {
    fprintf(stderr, "Usage: %s [--all] <circuit.r1cs> <witness.wtns> [more.wtns ...]\n", prog);
    return 1;
  }
  std::vector<uint8_t> r1cs_bytes;
  if (!read_file(argv[1], r1cs_bytes)) { fprintf(stderr, "Failed to read %s\n", argv[1]); return 1; }
  gw_status_t st; st.code = OK; st.error_msg = nullptr;
  gw_r1cs_t* r = nullptr;
  if (gw_r1cs_load(r1cs_bytes.data(), r1cs_bytes.size(), &r, &st)) {
    fprintf(stderr, "Error: %s: %s\n", argv[1], st.error_msg ? st.error_msg : "unknown");
    gw_free_status(&st);
    return 1;
  }
  gw_r1cs_info_t info; gw_r1cs_info(r, &info);
  const size_t row_b = (size_t)info.n_wires * 32;
  const int n_files = argc - 2;
  std::vector<std::string> verdict(n_files);
  std::vector<int> slot(n_files, -1);
  std::vector<uint8_t> rows;
  size_t n_rows = 0;
  for (int i = 0; i < n_files; i++) {
    std::vector<uint8_t> b;
    size_t payload = 0;
    if (!read_file(argv[2 + i], b)) { verdict[i] = "cannot be read"; continue; }
    verdict[i] = parse_wtns(b, info.n_wires, &payload);
    if (!verdict[i].empty()) continue;
    rows.insert(rows.end(), b.begin() + payload, b.begin() + payload + row_b);
    slot[i] = (int)n_rows++;
  }
  std::vector<uint32_t> first_failed(n_rows);
  const size_t n_con = info.n_constraints, abc_b = 3 * 32 * n_con;
  std::vector<uint8_t> abc(all ? n_rows * abc_b : 0);
  if (n_rows && (all ? gw_r1cs_abc_batch(r, rows.data(), n_rows, row_b, abc.data(), abc_b, 0, first_failed.data(), 1, &st)
                     : gw_r1cs_check_batch(r, rows.data(), n_rows, row_b, first_failed.data(), 1, &st))) {
    fprintf(stderr, "Error: %s\n", st.error_msg ? st.error_msg : "unknown");
    gw_free_status(&st);
    gw_r1cs_free(r);
    return 1;
  }
  int bad = 0;
  for (int i = 0; i < n_files; i++) {
    if (slot[i] >= 0) verdict[i] = first_failed[slot[i]] == GW_R1CS_OK ? "OK" : "constraint " + std::to_string(first_failed[slot[i]]) + " not satisfied";
    bad += verdict[i] != "OK";
    printf("%s: %s\n", argv[2 + i], verdict[i].c_str());
    if (!all || slot[i] < 0 || first_failed[slot[i]] == GW_R1CS_OK) continue;
    const uint8_t* a = abc.data() + slot[i] * abc_b;
    for (size_t k = 0; k < n_con; k++) {
      const uint8_t *ak = a + 32 * k, *bk = ak + 32 * n_con, *ck = bk + 32 * n_con;
      if (!gw::r1cs_holds(to_fe(ak), to_fe(bk), to_fe(ck)))
        printf("  constraint %zu: %s * %s != %s\n", k, decimal(ak).c_str(), decimal(bk).c_str(), decimal(ck).c_str());
    }
    const uint8_t* w = rows.data() + slot[i] * row_b;
    for (uint32_t j = 0; j < info.n_wires; j++)
      if (gw::fe_geq_m(to_fe(w + 32 * (size_t)j))) printf("  wire %u: %s >= M\n", j, decimal(w + 32 * (size_t)j).c_str());
  }
  gw_r1cs_free(r);
  return bad ? 1 : 0;
}
