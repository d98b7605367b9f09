/* TEST-ONLY stand-in for libbpmsm.so, built on the oracle's CPU arithmetic (oracle/ge.h, sc.h, hashes.h).
 *
 * Purpose: the C++ host mirror of the reference API (bulletproofs_b200/host/: RangeProof, InnerProductProof, LinearProof, r1cs, mpc)
 * talks to the engine only through the C ABI of include/bpmsm.h.  Linking that mirror against this library instead lets the CPU test
 * tier exercise the mirror's own logic -- transcript order, scalar algebra, wire formats, which MSMs it asks for -- and compare the
 * bytes it produces with the oracle's, on a machine without a GPU (tests/test_host_mirror_cpu.py).  It also times the host side of the
 * mirror alone: every entry point adds its own duration to a counter (mock_engine_seconds).
 *
 * This is NOT a CPU fallback of the product: nothing in bulletproofs_b200/ builds, loads or links it; the package loads libbpmsm.so only
 * and every compute entry point of that library fails without an sm_100 device.  The entry points the mirror does not use are
 * stubs that return BP_ERR_CUDA.  Only tests/ may use this file (it includes oracle/ headers).
 *
 * Algorithms are the reference's own, literally (folded generators in the inner-product argument, one MSM per call): the engine's
 * unfolded / batched forms are checked against the oracle on the GPU tier, this file is not a check of the engine.
 */
#define _GNU_SOURCE
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include "../../oracle/ge.h"
#include "../../oracle/hashes.h"

#include "../../include/bpmsm.h"      /* the prototypes this file must match */
#define BP_POINT_DYNAMIC 0x80000000u

/* from liboracle.so */
extern void *orc_gens_new(size_t gens_capacity, size_t party_capacity);
extern void orc_gens_free(void *h);
extern void orc_gens_get(void *h, int which, size_t party, size_t idx, uint8_t out[32]);
extern void orc_pedersen_gens(uint8_t B[32], uint8_t Bb[32]);
extern int orc_rangeproof_verify(void *gens, const uint8_t *transcript_state, const uint8_t *proof, size_t plen, const uint8_t *Vs, size_t m, size_t n, const uint8_t *seed);

struct bp_ctx { char err[256]; };
struct bp_gens { void *og; size_t cap, parties, n_points; ge *tab; uint8_t *enc; };      /* [B_blinding, B, G[party][i].., H[party][i]..] */
struct bp_ipp { bp_ctx *ctx; size_t N; ge *G, *H; ge Q; };
struct bp_ippx { bp_ctx *ctx; size_t N, B, cur; int first; sc *a, *b, *Gf, *Hf; ge *G, *H, *Q; };

static double g_seconds = 0.0;
static double now_s(void) { struct timespec t; clock_gettime(CLOCK_MONOTONIC, &t); return t.tv_sec + 1e-9 * t.tv_nsec; }
#define TIMED_BEGIN double t0__ = now_s()
#define TIMED_END g_seconds += now_s() - t0__
double mock_engine_seconds(void) { return g_seconds; }
void mock_engine_reset(void) { g_seconds = 0.0; }

static int load_scalars(sc *out, const uint8_t *bytes, size_t n) {
    for (size_t i = 0; i < n; i++) if (!sc_from_canonical(&out[i], bytes + 32 * i)) return BP_ERR_NONCANONICAL_SCALAR;
    return BP_OK;
}

/* ---- context */
int bp_ctx_create(int device, void *stream, bp_ctx **out) { (void)device; (void)stream; if (!out) return BP_ERR_INVALID_ARGUMENT; ge_init_constants(); *out = calloc(1, sizeof(bp_ctx)); return *out ? BP_OK : BP_ERR_CUDA; }
void bp_ctx_destroy(bp_ctx *c) { free(c); }
const char *bp_last_error(const bp_ctx *c) { return c ? c->err : "null context"; }
uint64_t bp_ctx_launch_count(const bp_ctx *c) { (void)c; return 0; }
int bp_ctx_set_msm_window(bp_ctx *c, int w) { (void)c; (void)w; return BP_OK; }
int bp_ctx_synchronize(bp_ctx *c) { (void)c; return BP_OK; }

/* ---- transcripts: the oracle's merlin struct is the 203-byte wire state */
void bp_transcript_new(const uint8_t *label, size_t len, uint8_t state[BP_TRANSCRIPT_BYTES]) { merlin m; merlin_init(&m, label, len); memcpy(state, &m, BP_TRANSCRIPT_BYTES); }
void bp_transcript_append_message(uint8_t state[BP_TRANSCRIPT_BYTES], const char *label, const uint8_t *msg, size_t len) { merlin m; memcpy(&m, state, BP_TRANSCRIPT_BYTES); merlin_append(&m, label, msg, len); memcpy(state, &m, BP_TRANSCRIPT_BYTES); }
void bp_transcript_append_u64(uint8_t state[BP_TRANSCRIPT_BYTES], const char *label, uint64_t x) { merlin m; memcpy(&m, state, BP_TRANSCRIPT_BYTES); merlin_append_u64(&m, label, x); memcpy(state, &m, BP_TRANSCRIPT_BYTES); }
void bp_transcript_challenge_bytes(uint8_t state[BP_TRANSCRIPT_BYTES], const char *label, uint8_t *out, size_t len) { merlin m; memcpy(&m, state, BP_TRANSCRIPT_BYTES); merlin_challenge(&m, label, out, len); memcpy(state, &m, BP_TRANSCRIPT_BYTES); }

/* ---- generator table */
int bp_gens_create(bp_ctx *c, size_t cap, size_t parties, bp_gens **out) {
    if (!c || !out || cap == 0 || parties == 0) return BP_ERR_INVALID_ARGUMENT;
    TIMED_BEGIN;
    bp_gens *g = calloc(1, sizeof *g);
    g->og = orc_gens_new(cap, parties); g->cap = cap; g->parties = parties; g->n_points = 2 + 2 * cap * parties;
    g->tab = malloc(g->n_points * sizeof(ge)); g->enc = malloc(g->n_points * 32);
    orc_pedersen_gens(g->enc + 32, g->enc);                                  /* slot 0 = B_blinding, slot 1 = B */
    for (size_t p = 0; p < parties; p++)
        for (size_t i = 0; i < cap; i++) {
            orc_gens_get(g->og, 0, p, i, g->enc + 32 * (2 + p * cap + i));
            orc_gens_get(g->og, 1, p, i, g->enc + 32 * (2 + parties * cap + p * cap + i));
        }
    for (size_t t = 0; t < g->n_points; t++) ge_decode(&g->tab[t], g->enc + 32 * t);
    *out = g;
    TIMED_END;
    return BP_OK;
}
void bp_gens_destroy(bp_gens *g) { if (!g) return; orc_gens_free(g->og); free(g->tab); free(g->enc); free(g); }
int bp_gens_get(bp_gens *g, int which, size_t party, size_t index, uint8_t out[32]) {
    if (!g || !out) return BP_ERR_INVALID_ARGUMENT;
    size_t slot;
    if (which == 2) slot = 1; else if (which == 3) slot = 0;
    else { if (party >= g->parties || index >= g->cap || which < 0 || which > 1) return BP_ERR_INVALID_ARGUMENT; slot = 2 + (which ? g->parties * g->cap : 0) + party * g->cap + index; }
    memcpy(out, g->enc + 32 * slot, 32); return BP_OK;
}

/* ---- group primitives and MSMs */
int bp_decompress_check_batch(bp_ctx *c, const uint8_t *points, size_t n, uint8_t *ok) {
    if (!c || !points || !ok) return BP_ERR_INVALID_ARGUMENT;
    TIMED_BEGIN;
    for (size_t i = 0; i < n; i++) { ge p; ok[i] = ge_decode(&p, points + 32 * i) ? 1 : 0; }
    TIMED_END; return BP_OK;
}
/* BP_MOCK_SKIP_POINT_MATH=1 (tests/mock_engine/profile_mirror.py only): every point result is the first input point, so that a profile of
 * the mirror is not drowned in the mock's own curve arithmetic.  The outputs are then meaningless (proofs do not verify). */
static int skip_math(void) { static int f = -1; if (f < 0) f = getenv("BP_MOCK_SKIP_POINT_MATH") != NULL; return f; }
static void msm_ge(uint8_t out[32], const sc *s, const ge *p, size_t n) { ge r; if (skip_math() && n) r = p[0]; else ge_msm_vartime(&r, s, p, n); ge_encode(out, &r); }

int bp_msm_batch(bp_ctx *c, const uint8_t *scalars, const uint8_t *points, const uint64_t *offsets, size_t n_msm, uint8_t *outs, uint8_t *status) {
    if (!c || !offsets || !outs || n_msm == 0) return BP_ERR_INVALID_ARGUMENT;
    TIMED_BEGIN;
    for (size_t j = 0; j < n_msm; j++) {
        size_t lo = offsets[j], n = offsets[j + 1] - lo;
        sc *s = malloc((n + 1) * sizeof(sc)); ge *p = malloc((n + 1) * sizeof(ge));
        uint8_t st = load_scalars(s, scalars + 32 * lo, n);
        for (size_t i = 0; i < n && st == BP_OK; i++) if (!ge_decode(&p[i], points + 32 * (lo + i))) st = BP_ERR_INVALID_POINT;
        if (st == BP_OK) msm_ge(outs + 32 * j, s, p, n); else memset(outs + 32 * j, 0, 32);
        if (status) status[j] = st;
        free(s); free(p);
    }
    TIMED_END; return BP_OK;
}
int bp_msm(bp_ctx *c, const uint8_t *scalars, const uint8_t *points, size_t n, uint8_t out[32]) {
    uint64_t off[2] = {0, n}; uint8_t st = 0;
    int rc = bp_msm_batch(c, scalars, points, off, 1, out, &st);
    return rc ? rc : st;
}
int bp_msm_indexed_batch(bp_ctx *c, bp_gens *gens, const uint8_t *scalars, const uint32_t *point_idx, const uint8_t *dyn_points, size_t n_dyn,
                         const uint64_t *offsets, size_t n_msm, uint8_t *outs, uint8_t *status) {
    if (!c || !offsets || !outs || n_msm == 0 || !scalars || !point_idx || offsets[0] != 0 || offsets[n_msm] == 0) return BP_ERR_INVALID_ARGUMENT;
    TIMED_BEGIN;
    size_t T = offsets[n_msm];
    for (size_t t = 0; t < T; t++) {
        uint32_t v = point_idx[t];
        if (v & BP_POINT_DYNAMIC) { if ((v & 0x7fffffffu) >= n_dyn || !dyn_points) { TIMED_END; return BP_ERR_INVALID_ARGUMENT; } }
        else if (!gens || v >= gens->n_points) { TIMED_END; return BP_ERR_INVALID_ARGUMENT; }
    }
    ge *dyn = malloc((n_dyn + 1) * sizeof(ge)); uint8_t *dyn_ok = malloc(n_dyn + 1);
    for (size_t i = 0; i < n_dyn; i++) dyn_ok[i] = ge_decode(&dyn[i], dyn_points + 32 * i) ? 1 : 0;
    for (size_t j = 0; j < n_msm; j++) {
        size_t lo = offsets[j], n = offsets[j + 1] - lo;
        sc *s = malloc((n + 1) * sizeof(sc)); ge *p = malloc((n + 1) * sizeof(ge));
        uint8_t st = load_scalars(s, scalars + 32 * lo, n);
        for (size_t i = 0; i < n; i++) {
            uint32_t v = point_idx[lo + i];
            if (v & BP_POINT_DYNAMIC) { uint32_t d = v & 0x7fffffffu; if (!dyn_ok[d]) { if (st == BP_OK) st = BP_ERR_INVALID_POINT; ge_identity(&p[i]); } else p[i] = dyn[d]; }
            else p[i] = gens->tab[v];
        }
        if (st == BP_OK) msm_ge(outs + 32 * j, s, p, n); else memset(outs + 32 * j, 0, 32);
        if (status) status[j] = st;
        free(s); free(p);
    }
    free(dyn); free(dyn_ok);
    TIMED_END; return BP_OK;
}

/* ---- inner-product argument, folding form (inner_product_proof.rs:87-178 as LinearProof uses it through the mirror) */
static int ipp_new(bp_ctx *c, size_t N, bp_ipp **out) {
    if (!c || !out || N == 0 || (N & (N - 1))) return BP_ERR_INVALID_ARGUMENT;
    bp_ipp *s = calloc(1, sizeof *s); s->ctx = c; s->N = N; s->G = malloc(N * sizeof(ge)); s->H = malloc(N * sizeof(ge)); *out = s; return BP_OK;
}
void bp_ipp_end(bp_ipp *s) { if (!s) return; free(s->G); free(s->H); free(s); }
int bp_ipp_begin_points(bp_ctx *c, const uint8_t *G, const uint8_t *H, size_t N, const uint8_t Q[32], bp_ipp **out) {
    if (!G || !H || !Q) return BP_ERR_INVALID_ARGUMENT;
    int rc = ipp_new(c, N, out); if (rc) return rc;
    TIMED_BEGIN;
    bp_ipp *s = *out; int ok = ge_decode(&s->Q, Q);
    for (size_t i = 0; i < N; i++) ok &= ge_decode(&s->G[i], G + 32 * i) & ge_decode(&s->H[i], H + 32 * i);
    TIMED_END;
    if (!ok) { bp_ipp_end(s); *out = NULL; return BP_ERR_INVALID_POINT; }
    return BP_OK;
}
int bp_ipp_lr(bp_ipp *s, size_t h, const uint8_t *sL, const uint8_t *sR, uint8_t L_out[32], uint8_t R_out[32]) {
    if (!s || !sL || !sR || !L_out || !R_out || h == 0 || 2 * h > s->N) return BP_ERR_INVALID_ARGUMENT;
    TIMED_BEGIN;
    size_t n = 2 * h + 1; sc *sc_ = malloc(n * sizeof(sc)); ge *p = malloc(n * sizeof(ge)); int rc;
    if ((rc = load_scalars(sc_, sL, n)) == BP_OK) {
        for (size_t i = 0; i < h; i++) { p[i] = s->G[h + i]; p[h + i] = s->H[i]; }
        p[2 * h] = s->Q; msm_ge(L_out, sc_, p, n);
        if ((rc = load_scalars(sc_, sR, n)) == BP_OK) {
            for (size_t i = 0; i < h; i++) { p[i] = s->G[i]; p[h + i] = s->H[h + i]; }
            msm_ge(R_out, sc_, p, n);
        }
    }
    free(sc_); free(p);
    TIMED_END; return rc;
}
static void lincomb2(ge *out, const sc *x, const ge *P, const sc *y, const ge *Q) { if (skip_math()) { *out = *P; return; } sc s[2] = {*x, *y}; ge p[2] = {*P, *Q}; ge_msm_vartime(out, s, p, 2); }
int bp_ipp_fold(bp_ipp *s, size_t h, const uint8_t *g_lo, const uint8_t *g_hi, const uint8_t *h_lo, const uint8_t *h_hi, int per_index) {
    if (!s || !g_lo || !g_hi || !h_lo || !h_hi || h == 0 || 2 * h > s->N) return BP_ERR_INVALID_ARGUMENT;
    TIMED_BEGIN;
    int rc = BP_OK;
    for (size_t i = 0; i < h && rc == BP_OK; i++) {
        size_t k = per_index ? i : 0; sc a, b, c2, d;
        if (!sc_from_canonical(&a, g_lo + 32 * k) || !sc_from_canonical(&b, g_hi + 32 * k) || !sc_from_canonical(&c2, h_lo + 32 * k) || !sc_from_canonical(&d, h_hi + 32 * k)) { rc = BP_ERR_NONCANONICAL_SCALAR; break; }
        ge g, hh; lincomb2(&g, &a, &s->G[i], &b, &s->G[h + i]); lincomb2(&hh, &c2, &s->H[i], &d, &s->H[h + i]);
        s->G[i] = g; s->H[i] = hh;
    }
    TIMED_END; return rc;       /* as in the engine, the session keeps its original capacity: the caller addresses halves by n_half */
}

/* ---- InnerProductProof::create as a session (inner_product_proof.rs:38-193), n_proofs proofs side by side, folding form */
void bp_ippx_end(bp_ippx *s) { if (!s) return; free(s->a); free(s->b); free(s->Gf); free(s->Hf); free(s->G); free(s->H); free(s->Q); free(s); }
static int ippx_new(bp_ctx *c, size_t N, size_t B, const uint8_t *Q, const uint8_t *Gf, const uint8_t *Hf, const uint8_t *a, const uint8_t *b, bp_ippx **out) {
    if (!c || !out || !Q || !a || !b || N == 0 || (N & (N - 1)) || B == 0) return BP_ERR_INVALID_ARGUMENT;
    bp_ippx *s = calloc(1, sizeof *s); s->ctx = c; s->N = s->cur = N; s->B = B; s->first = 1;
    size_t BN = B * N;
    s->a = malloc(BN * sizeof(sc)); s->b = malloc(BN * sizeof(sc)); s->Gf = malloc(BN * sizeof(sc)); s->Hf = malloc(BN * sizeof(sc));
    s->G = malloc(BN * sizeof(ge)); s->H = malloc(BN * sizeof(ge)); s->Q = malloc(B * sizeof(ge));
    int rc = load_scalars(s->a, a, BN); if (!rc) rc = load_scalars(s->b, b, BN);
    sc one; sc_from_u64(&one, 1);
    if (!rc) { if (Gf) rc = load_scalars(s->Gf, Gf, BN); else for (size_t i = 0; i < BN; i++) s->Gf[i] = one; }
    if (!rc) { if (Hf) rc = load_scalars(s->Hf, Hf, BN); else for (size_t i = 0; i < BN; i++) s->Hf[i] = one; }
    for (size_t p = 0; p < B && !rc; p++) if (!ge_decode(&s->Q[p], Q + 32 * p)) rc = BP_ERR_INVALID_POINT;
    if (rc) { bp_ippx_end(s); return rc; }
    *out = s; return BP_OK;
}
int bp_ippx_begin(bp_ctx *c, bp_gens *gens, size_t n, size_t m, size_t B, const uint8_t *Q, const uint8_t *Gf, const uint8_t *Hf, const uint8_t *a, const uint8_t *b, bp_ippx **out) {
    if (!gens || n == 0 || m == 0 || n > gens->cap || m > gens->parties) return BP_ERR_INVALID_ARGUMENT;
    TIMED_BEGIN;
    int rc = ippx_new(c, n * m, B, Q, Gf, Hf, a, b, out);
    if (!rc) { bp_ippx *s = *out; size_t N = n * m;
        for (size_t p = 0; p < B; p++) for (size_t q = 0; q < N; q++) {
            s->G[p * N + q] = gens->tab[2 + (q / n) * gens->cap + q % n]; s->H[p * N + q] = gens->tab[2 + gens->parties * gens->cap + (q / n) * gens->cap + q % n]; } }
    TIMED_END; return rc;
}
int bp_ippx_begin_points(bp_ctx *c, const uint8_t *G, const uint8_t *H, size_t N, size_t B, const uint8_t *Q, const uint8_t *Gf, const uint8_t *Hf, const uint8_t *a, const uint8_t *b, bp_ippx **out) {
    if (!G || !H) return BP_ERR_INVALID_ARGUMENT;
    TIMED_BEGIN;
    int rc = ippx_new(c, N, B, Q, Gf, Hf, a, b, out);
    if (!rc) { bp_ippx *s = *out; int ok = 1;
        for (size_t q = 0; q < N; q++) { ok &= ge_decode(&s->G[q], G + 32 * q) & ge_decode(&s->H[q], H + 32 * q); }
        for (size_t p = 1; p < B; p++) { memcpy(s->G + p * N, s->G, N * sizeof(ge)); memcpy(s->H + p * N, s->H, N * sizeof(ge)); }
        if (!ok) { bp_ippx_end(s); *out = NULL; rc = BP_ERR_INVALID_POINT; } }
    TIMED_END; return rc;
}
size_t bp_ippx_current_len(const bp_ippx *s) { return s ? s->cur : 0; }
int bp_ippx_round(bp_ippx *s, uint8_t *LR_out) {
    if (!s || !LR_out || s->cur < 2) return BP_ERR_INVALID_ARGUMENT;
    TIMED_BEGIN;
    size_t h = s->cur / 2, n = 2 * h + 1; sc *w = malloc(n * sizeof(sc)); ge *p = malloc(n * sizeof(ge));
    for (size_t q = 0; q < s->B; q++) {
        sc *a = s->a + q * s->N, *b = s->b + q * s->N, *gf = s->Gf + q * s->N, *hf = s->Hf + q * s->N; ge *G = s->G + q * s->N, *H = s->H + q * s->N;
        sc cL, cR, t; sc_zero(&cL); sc_zero(&cR);
        for (size_t i = 0; i < h; i++) { sc_mul(&t, &a[i], &b[h + i]); sc_add(&cL, &cL, &t); sc_mul(&t, &a[h + i], &b[i]); sc_add(&cR, &cR, &t); }
        for (size_t i = 0; i < h; i++) {                 /* L: a_L * G_R (factors of G_R), b_R * H_L (factors of H_L), c_L Q   (:87-99 / :153-158) */
            if (s->first) { sc_mul(&w[i], &a[i], &gf[h + i]); sc_mul(&w[h + i], &b[h + i], &hf[i]); } else { w[i] = a[i]; w[h + i] = b[h + i]; }
            p[i] = G[h + i]; p[h + i] = H[i];
        }
        w[2 * h] = cL; p[2 * h] = s->Q[q]; msm_ge(LR_out + 64 * q, w, p, n);
        for (size_t i = 0; i < h; i++) {                 /* R: a_R * G_L, b_L * H_R, c_R Q   (:101-113 / :159-163) */
            if (s->first) { sc_mul(&w[i], &a[h + i], &gf[i]); sc_mul(&w[h + i], &b[i], &hf[h + i]); } else { w[i] = a[h + i]; w[h + i] = b[i]; }
            p[i] = G[i]; p[h + i] = H[h + i];
        }
        w[2 * h] = cR; msm_ge(LR_out + 64 * q + 32, w, p, n);
    }
    free(w); free(p);
    TIMED_END; return BP_OK;
}
int bp_ippx_fold(bp_ippx *s, const uint8_t *u_bytes, const uint8_t *ui_bytes) {
    if (!s || !u_bytes || !ui_bytes || s->cur < 2) return BP_ERR_INVALID_ARGUMENT;
    TIMED_BEGIN;
    size_t h = s->cur / 2; int rc = BP_OK;
    for (size_t q = 0; q < s->B && rc == BP_OK; q++) {
        sc u, ui, t, x, y;
        if (!sc_from_canonical(&u, u_bytes + 32 * q) || !sc_from_canonical(&ui, ui_bytes + 32 * q)) { rc = BP_ERR_NONCANONICAL_SCALAR; break; }
        sc *a = s->a + q * s->N, *b = s->b + q * s->N, *gf = s->Gf + q * s->N, *hf = s->Hf + q * s->N; ge *G = s->G + q * s->N, *H = s->H + q * s->N;
        for (size_t i = 0; i < h; i++) {                 /* :122-134 (first round, factors folded in) / :172-178 */
            sc_mul(&t, &a[i], &u); sc_mul(&x, &ui, &a[h + i]); sc_add(&a[i], &t, &x);
            sc_mul(&t, &b[i], &ui); sc_mul(&x, &u, &b[h + i]); sc_add(&b[i], &t, &x);
            ge g, hh;
            if (s->first) { sc_mul(&x, &ui, &gf[i]); sc_mul(&y, &u, &gf[h + i]); lincomb2(&g, &x, &G[i], &y, &G[h + i]); sc_mul(&x, &u, &hf[i]); sc_mul(&y, &ui, &hf[h + i]); lincomb2(&hh, &x, &H[i], &y, &H[h + i]); }
            else { lincomb2(&g, &ui, &G[i], &u, &G[h + i]); lincomb2(&hh, &u, &H[i], &ui, &H[h + i]); }
            G[i] = g; H[i] = hh;
        }
    }
    s->cur = h; s->first = 0;
    TIMED_END; return rc;
}
int bp_ippx_finish(bp_ippx *s, uint8_t *ab_out) {
    if (!s || !ab_out || s->cur != 1) return BP_ERR_INVALID_ARGUMENT;
    for (size_t q = 0; q < s->B; q++) { sc_tobytes(ab_out + 64 * q, &s->a[q * s->N]); sc_tobytes(ab_out + 64 * q + 32, &s->b[q * s->N]); }
    return BP_OK;
}

/* ---- range-proof verification: the oracle's per-proof verify_multiple */
int bp_rangeproof_verify_batch(bp_ctx *c, bp_gens *gens, const uint8_t *transcript, const uint8_t *proofs, size_t proof_len, const uint8_t *commitments,
                               size_t n, size_t m, size_t count, const uint8_t *seed, uint8_t *verdicts) {
    if (!c || !gens || !transcript || !proofs || !commitments || !verdicts || count == 0) return BP_ERR_INVALID_ARGUMENT;
    TIMED_BEGIN;
    uint8_t zero[32] = {0};
    for (size_t i = 0; i < count; i++) verdicts[i] = (uint8_t)orc_rangeproof_verify(gens->og, transcript, proofs + i * proof_len, proof_len, commitments + 32 * m * i, m, n, seed ? seed : zero);
    TIMED_END; return BP_OK;
}

