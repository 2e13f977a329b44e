/* calc_witness <inputs.json> <graph.bin> <witness.wtns>
 *
 * Embedding example of the drop-in C ABI (include/graph_witness.h, part 1 only), in plain C and with the argument
 * order of circom-witnesscalc's examples/calc_witness.c: read the inputs JSON and the wtns.graph.001 file, call
 * gw_calc_witness, write the .wtns file it returns.  Like the reference's example it trusts the return value, not
 * status.code.  build.py compiles it as bin/example-calc-witness; the tests compare what it writes with the golden
 * .wtns files.
 */
#include <stdio.h>
#include <stdlib.h>

#include "../include/graph_witness.h"

/* whole file into a malloc'ed buffer with one extra NUL byte (the inputs are passed as a C string) */
static char *read_file(const char *path, size_t *len) {
  FILE *f = fopen(path, "rb");
  if (f == NULL) return NULL;
  char *buf = NULL;
  long n = -1;
  if (fseek(f, 0, SEEK_END) == 0) n = ftell(f);
  if (n >= 0 && fseek(f, 0, SEEK_SET) == 0) buf = malloc((size_t)n + 1);
  if (buf != NULL && fread(buf, 1, (size_t)n, f) != (size_t)n) {
    free(buf);
    buf = NULL;
  }
  fclose(f);
  if (buf != NULL) {
    buf[n] = '\0';
    *len = (size_t)n;
  }
  return buf;
}

int main(int argc, char *argv[]) {
  if (argc != 4) {
    fprintf(stderr, "Usage: %s <inputs.json> <graph.bin> <witness.wtns>\n", argv[0]);
    return 1;
  }
  size_t inputs_len = 0, graph_len = 0;
  char *inputs = read_file(argv[1], &inputs_len);
  if (inputs == NULL) {
    fprintf(stderr, "cannot read %s\n", argv[1]);
    return 1;
  }
  char *graph = read_file(argv[2], &graph_len);
  if (graph == NULL) {
    fprintf(stderr, "cannot read %s\n", argv[2]);
    free(inputs);
    return 1;
  }

  gw_status_t status = {OK, NULL};
  void *wtns = NULL;
  size_t wtns_len = 0;
  int rc = gw_calc_witness(inputs, graph, graph_len, &wtns, &wtns_len, &status);
  free(inputs);
  free(graph);
  if (rc != 0) {
    fprintf(stderr, "Error: %s\n", status.error_msg != NULL ? status.error_msg : "unknown");
    gw_free_status(&status);
    return 1;
  }

  FILE *out = fopen(argv[3], "wb");
  int ok = out != NULL && fwrite(wtns, 1, wtns_len, out) == wtns_len;
  if (out != NULL && fclose(out) != 0) ok = 0;
  free(wtns);
  if (!ok) {
    fprintf(stderr, "cannot write %s\n", argv[3]);
    return 1;
  }
  printf("witness saved to %s (%zu bytes)\n", argv[3], wtns_len);
  return 0;
}
