/* TEST-ONLY: bp_msm_indexed_batch_ct and a call log on top of the mock engine (mock_bpmsm.c), for the routing checks of
 * tests/test_msm_ct_cpu.py.  That test links the mock engine, this file and the C++ host mirror (built with -DBP_HOST_REQUIRE_CT, as
 * the library build does) into one library in a temporary directory, with -Wl,--wrap for the variable-time MSM entry points, so that
 * every MSM the mirror asks for is recorded: entry point, point indices, offsets, scalars.
 *
 * The ct entry point here computes with the mock's (variable-time) oracle arithmetic: what is under test is which entry point the
 * mirror calls and with which public arguments, not the engine's timing. */
#include <stdlib.h>
#include <string.h>
#include "../../include/bpmsm_ct.h"

int __real_bp_msm_indexed_batch(bp_ctx *c, bp_gens *gens, const uint8_t *scalars, const uint32_t *point_idx, const uint8_t *dyn_points, size_t n_dyn,
                                const uint64_t *offsets, size_t n_msm, uint8_t *outs, uint8_t *status);
int __real_bp_msm_batch(bp_ctx *c, const uint8_t *scalars, const uint8_t *points, const uint64_t *offsets, size_t n_msm, uint8_t *outs, uint8_t *status);

typedef struct { const char *name; size_t n_terms, n_msm; uint32_t *idx; uint64_t *offsets; uint8_t *scalars; } log_entry;
static log_entry *g_log = NULL;
static size_t g_log_n = 0, g_log_cap = 0;

void ct_log_reset(void) {
    for (size_t i = 0; i < g_log_n; i++) { free(g_log[i].idx); free(g_log[i].offsets); free(g_log[i].scalars); }
    g_log_n = 0;
}
size_t ct_log_count(void) { return g_log_n; }
/* entry i: returns its name; n_terms / n_msm out; idx / offsets / scalars copied out when non-NULL (n_terms, n_msm + 1, 32 * n_terms words / bytes) */
const char *ct_log_entry(size_t i, size_t *n_terms, size_t *n_msm, uint32_t *idx, uint64_t *offsets, uint8_t *scalars) {
    if (i >= g_log_n) return NULL;
    const log_entry *e = &g_log[i];
    *n_terms = e->n_terms; *n_msm = e->n_msm;
    if (idx && e->idx) memcpy(idx, e->idx, 4 * e->n_terms);
    if (offsets) memcpy(offsets, e->offsets, 8 * (e->n_msm + 1));
    if (scalars) memcpy(scalars, e->scalars, 32 * e->n_terms);
    return e->name;
}
static void log_call(const char *name, const uint8_t *scalars, const uint32_t *idx, const uint64_t *offsets, size_t n_msm) {
    if (!offsets || n_msm == 0 || !scalars) return;
    if (g_log_n == g_log_cap) { g_log_cap = g_log_cap ? 2 * g_log_cap : 64; g_log = realloc(g_log, g_log_cap * sizeof *g_log); }
    size_t T = offsets[n_msm];
    log_entry *e = &g_log[g_log_n++];
    e->name = name; e->n_terms = T; e->n_msm = n_msm;
    e->idx = NULL;
    if (idx) { e->idx = malloc(4 * T + 4); memcpy(e->idx, idx, 4 * T); }
    e->offsets = malloc(8 * (n_msm + 1)); memcpy(e->offsets, offsets, 8 * (n_msm + 1));
    e->scalars = malloc(32 * T + 32); memcpy(e->scalars, scalars, 32 * T);
}

int bp_msm_indexed_batch_ct(bp_ctx *c, bp_gens *gens, const uint8_t *scalars, const uint32_t *point_idx, const uint64_t *offsets, size_t n_msm,
                            uint8_t *outs, uint8_t *status) {
    if (!gens) return BP_ERR_INVALID_ARGUMENT;
    log_call("bp_msm_indexed_batch_ct", scalars, point_idx, offsets, n_msm);
    return __real_bp_msm_indexed_batch(c, gens, scalars, point_idx, NULL, 0, offsets, n_msm, outs, status);
}
int __wrap_bp_msm_indexed_batch(bp_ctx *c, bp_gens *gens, const uint8_t *scalars, const uint32_t *point_idx, const uint8_t *dyn_points, size_t n_dyn,
                                const uint64_t *offsets, size_t n_msm, uint8_t *outs, uint8_t *status) {
    log_call("bp_msm_indexed_batch", scalars, point_idx, offsets, n_msm);
    return __real_bp_msm_indexed_batch(c, gens, scalars, point_idx, dyn_points, n_dyn, offsets, n_msm, outs, status);
}
int __wrap_bp_msm_batch(bp_ctx *c, const uint8_t *scalars, const uint8_t *points, const uint64_t *offsets, size_t n_msm, uint8_t *outs, uint8_t *status) {
    log_call("bp_msm_batch", scalars, NULL, offsets, n_msm);
    return __real_bp_msm_batch(c, scalars, points, offsets, n_msm, outs, status);
}
