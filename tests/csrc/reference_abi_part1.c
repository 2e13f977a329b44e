/* Part 1 of include/graph_witness.h against the drop-in ABI of circom-witnesscalc's own header
 * (include/graph_witness.h:7-28 there), whose declarations SURVEY.md section 8(b) records:
 *
 *   typedef enum {OK=0, ERROR=1} GW_ERROR_CODE;
 *   typedef struct {GW_ERROR_CODE code; char *error_msg;} gw_status_t;
 *   int gw_calc_witness(const char *inputs, const void *graph_data, const size_t graph_data_len,
 *                       void **wtns_data, size_t *wtns_len, const gw_status_t *status);
 *   void gw_free_status(gw_status_t *status);
 *
 * They are restated below under ref_ names, and this file compiles (C11, -Werror) only if this project's header
 * declares the same constants, the same layout and field types, and functions of the same types.
 * tests/test_cabi.py compiles it.
 */
#include <stddef.h>

#include "../../include/graph_witness.h"

typedef enum { REF_OK = 0, REF_ERROR = 1 } ref_GW_ERROR_CODE;
typedef struct {
  ref_GW_ERROR_CODE code;
  char *error_msg;
} ref_gw_status_t;

_Static_assert((int)OK == (int)REF_OK && (int)ERROR == (int)REF_ERROR, "GW_ERROR_CODE constants");
_Static_assert(sizeof(GW_ERROR_CODE) == sizeof(ref_GW_ERROR_CODE), "GW_ERROR_CODE size");
_Static_assert(sizeof(gw_status_t) == sizeof(ref_gw_status_t), "gw_status_t size");
_Static_assert(offsetof(gw_status_t, code) == offsetof(ref_gw_status_t, code), "gw_status_t.code offset");
_Static_assert(offsetof(gw_status_t, error_msg) == offsetof(ref_gw_status_t, error_msg), "gw_status_t.error_msg offset");

/* field types: a pointer of another type is an incompatible-pointer-types diagnostic, an error under -Werror */
void ref_abi_fields(gw_status_t *s, GW_ERROR_CODE **code, char ***error_msg) {
  *code = &s->code;
  *error_msg = &s->error_msg;
}

/* function types: the same assignment rule */
int (*const ref_abi_calc_witness)(const char *, const void *, const size_t, void **, size_t *,
                                  const gw_status_t *) = gw_calc_witness;
void (*const ref_abi_free_status)(gw_status_t *) = gw_free_status;
