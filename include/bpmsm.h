/* bpmsm.h — C ABI of the B200-native Ristretto255 multiscalar-multiplication engine.
 *
 * This is the drop-in boundary for the MSM-bound hot path of dalek-cryptography/bulletproofs.
 * The reference has no FFI; its only seam is the Rust trait surface of curve25519_dalek::traits
 * that the crate calls.  Each entry point below names the reference call site it replaces; the
 * Rust-side binding a maintainer would add is shown in INTEGRATION.md.
 *
 * Wire types (SURVEY.md §8b):
 *   scalar            32 bytes, little-endian, canonical (< l)          = curve25519_dalek::scalar::Scalar::as_bytes()
 *   compressed point  32 bytes, canonical Ristretto255 encoding         = CompressedRistretto::as_bytes()
 *   transcript        203 bytes: STROBE-128 state (200) ‖ pos ‖ pos_begin ‖ cur_flags  = merlin::Transcript fields
 *
 * Ownership: the caller owns every host buffer for the duration of the call; the library copies
 * in and out and retains nothing except the explicit handles (bp_ctx, bp_gens).
 * Threading: a bp_ctx is one device + one CUDA stream and is not thread-safe; different
 * contexts may be used concurrently.  There is no hidden global state and no CPU fallback:
 * every call fails with BP_ERR_CUDA when no sm_100 device is usable.
 * Timing: bp_msm_indexed_batch_ct (include/bpmsm_ct.h) is constant-time in its scalars: which kernels run, their grids, every memory address and every
 * copy depend only on the term count, the offsets and the point indices, and the only scalar-derived value it returns besides the
 * results is the per-MSM canonicality status.  Its point indices, offsets and results are public.  Every other entry point is
 * variable-time in all of its inputs, like the reference's vartime_* calls: use them for public data (verification, challenges)
 * only.  The C++ host mirror routes the reference's constant-time `multiscalar_mul` sites through the ct entry point; see
 * DESIGN.md "constant-time policy" for what is and is not covered.
 */
#ifndef BPMSM_H
#define BPMSM_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* call status */
#define BP_OK 0
#define BP_ERR_INVALID_POINT 1        /* a point failed to decompress: optional_multiscalar_mul -> None (range_proof/mod.rs:445) */
#define BP_ERR_LENGTH_MISMATCH 2      /* the reference panics (assert_eq!, inner_product_proof.rs:59-67) */
#define BP_ERR_NONCANONICAL_SCALAR 3  /* scalar bytes >= l: Scalar::from_canonical_bytes -> None */
#define BP_ERR_CUDA 4                 /* no device / launch failure; bp_last_error() has the text */
#define BP_ERR_INVALID_ARGUMENT 5

/* per-proof verdicts = ProofError variants (/root/reference/src/errors.rs:12-54) */
#define BP_PROOF_OK 0
#define BP_PROOF_VERIFICATION_ERROR 1
#define BP_PROOF_FORMAT_ERROR 2
#define BP_PROOF_INVALID_BITSIZE 3
#define BP_PROOF_INVALID_GENERATORS_LENGTH 4
#define BP_PROOF_INVALID_AGGREGATION 5

#define BP_TRANSCRIPT_BYTES 203

typedef struct bp_ctx bp_ctx;
typedef struct bp_gens bp_gens;

/* ---- context ------------------------------------------------------------------------------- */
/* stream: a cudaStream_t to run on (e.g. torch.cuda.current_stream().cuda_stream), or NULL to
 * create a private non-blocking stream. */
int bp_ctx_create(int device, void *stream, bp_ctx **out);
void bp_ctx_destroy(bp_ctx *ctx);
const char *bp_last_error(const bp_ctx *ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
uint64_t bp_ctx_launch_count(const bp_ctx *ctx);
/* Pippenger window size (bits) of the generic MSM entry points on this context: 0 = chosen by terms per MSM (default), 2..18 = fixed.
 * Results do not depend on it; tests use it to cover every window geometry, benchmarks to tune. */
int bp_ctx_set_msm_window(bp_ctx *ctx, int window_bits);
/* block until all work queued on the context's stream is finished */
int bp_ctx_synchronize(bp_ctx *ctx);

/* ---- group primitives ---------------------------------------------------------------------- */
/* CompressedRistretto::decompress for n points: ok[i] = 1 if point i is a valid encoding.
 * Replaces the inline decompress() calls of range_proof/mod.rs:433-443. */
int bp_decompress_check_batch(bp_ctx *ctx, const uint8_t *points, size_t n, uint8_t *ok);
/* RistrettoPoint::from_uniform_bytes (generators.rs:94-99) for n 64-byte inputs -> n compressed points */
int bp_from_uniform_bytes_batch(bp_ctx *ctx, const uint8_t *uniform, size_t n, uint8_t *points_out);

/* ---- multiscalar multiplication ------------------------------------------------------------ */
/* RistrettoPoint::vartime_multiscalar_mul / optional_multiscalar_mul on wire types:
 *   out = compress( sum_i scalars[i] * decompress(points[i]) ).
 * Call sites replaced: inner_product_proof.rs:87,101,127,131,153,159,177,178,308;
 * range_proof/mod.rs:421; range_proof/messages.rs:128,149.
 * Returns BP_ERR_INVALID_POINT if any point does not decode (the reference's `None`). */
int bp_msm(bp_ctx *ctx, const uint8_t *scalars, const uint8_t *points, size_t n, uint8_t out[32]);
/* n_msm independent MSMs in one launch sequence: MSM j uses terms offsets[j] .. offsets[j+1]-1.
 * outs = n_msm x 32 bytes; status[j] = BP_OK / BP_ERR_INVALID_POINT / BP_ERR_NONCANONICAL_SCALAR. */
int bp_msm_batch(bp_ctx *ctx, const uint8_t *scalars, const uint8_t *points, const uint64_t *offsets,
                 size_t n_msm, uint8_t *outs, uint8_t *status);
/* Same with every array already resident in device memory (16-byte aligned device pointers);
 * work is queued on the context's stream and the call returns without synchronising. */
int bp_msm_batch_device(bp_ctx *ctx, const void *d_scalars, const void *d_points, const void *d_offsets_u32,
                        size_t n_msm, size_t total_terms, void *d_outs, void *d_status);

/* MSMs whose points are generator-table entries and/or caller-supplied compressed points:
 * point_idx[t] < 2^31 selects table slot point_idx[t] of `gens` (layout of bp_gens_device_table: 0 = B_blinding,
 * 1 = B, 2 + party*cap + i = G[party][i], 2 + parties*cap + party*cap + i = H[party][i]); point_idx[t] = 2^31 | j
 * selects dyn_points[j].  This is how the public-scalar constant-base call sites run without re-uploading the table: Q = w*B
 * (dealer.rs:256), ProofShare::audit_share (messages.rs:128,149) and the R1CS verifier's mega-check.  The prover's commitments to
 * secrets (PedersenGens::commit, A, S, T_1/T_2) use bp_msm_indexed_batch_ct (include/bpmsm_ct.h). */
int bp_msm_indexed_batch(bp_ctx *ctx, bp_gens *gens, const uint8_t *scalars, const uint32_t *point_idx,
                         const uint8_t *dyn_points, size_t n_dyn, const uint64_t *offsets, size_t n_msm,
                         uint8_t *outs, uint8_t *status);

/* ---- inner-product argument, prover side, folding form ---------------------------------------- */
/* The generator vectors G, H (and Q) live on the device for the k rounds and are folded there; the host keeps the transcript and
 * the scalar vectors a, b and calls once per round for L,R and once for the fold.  This is the form LinearProof::create
 * (linear_proof.rs:40-160) runs on, with its own G and H vectors; InnerProductProof::create (inner_product_proof.rs:38-193) uses
 * the bp_ippx_* session below, which keeps a and b on the device as well and never folds a point. */
typedef struct bp_ipp bp_ipp;
/* G, H = N compressed points each (the reference's Vec<RistrettoPoint> arguments), Q compressed */
int bp_ipp_begin_points(bp_ctx *ctx, const uint8_t *G, const uint8_t *H, size_t N, const uint8_t Q[32], bp_ipp **out);
/* L = <sL[0..h), G_R> + <sL[h..2h), H_L> + sL[2h] Q,  R = <sR[0..h), G_L> + <sR[h..2h), H_R> + sR[2h] Q  (lines 87-113 / 153-163) */
int bp_ipp_lr(bp_ipp *sess, size_t n_half, const uint8_t *scalars_L, const uint8_t *scalars_R, uint8_t L_out[32], uint8_t R_out[32]);
/* G_L[i] = g_lo G_L[i] + g_hi G_R[i], H_L[i] = h_lo H_L[i] + h_hi H_R[i]  (lines 127-134 / 177-178);
 * per_index = 1: n_half scalars per array (first round, factors folded in), 0: one scalar per array */
int bp_ipp_fold(bp_ipp *sess, size_t n_half, const uint8_t *g_lo, const uint8_t *g_hi, const uint8_t *h_lo, const uint8_t *h_hi, int per_index);
void bp_ipp_end(bp_ipp *sess);

/* ---- point values across the boundary ------------------------------------------------------- */
/* CompressedRistretto::decompress() -> Option<RistrettoPoint> for n points (call sites src/range_proof/mod.rs:433-443,
 * src/inner_product_proof.rs:296-306, src/r1cs/verifier.rs:482): xyzt_out[i] = the extended coordinates X | Y | Z | T of point i as
 * four canonical 32-byte field elements (Z = 1) -- an in-memory RistrettoPoint a host caller can keep; ok[i] = 0 where the
 * reference would return None (the slot then holds the identity).  bp_compress_batch is RistrettoPoint::compress()
 * (src/inner_product_proof.rs:99,113, src/range_proof/dealer.rs:113-116) on such values (any projective representative). */
int bp_decompress_batch(bp_ctx *ctx, const uint8_t *points, size_t n, uint8_t *xyzt_out, uint8_t *ok);
int bp_compress_batch(bp_ctx *ctx, const uint8_t *xyzt, size_t n, uint8_t *points_out);

/* ---- resident point sets ------------------------------------------------------------------- */
/* A vector of n points decompressed once and kept on the device (affine Niels form, 96 B/point): the bases of repeated MSMs
 * (`Vec<RistrettoPoint>` reused across vartime_multiscalar_mul calls, e.g. the generator vectors of inner_product_proof.rs:87-178).
 * BP_ERR_INVALID_POINT if any encoding is invalid. */
typedef struct bp_points bp_points;
int bp_points_create(bp_ctx *ctx, const uint8_t *points, size_t n, bp_points **out);
int bp_points_create_device(bp_ctx *ctx, const void *d_points, size_t n, bp_points **out);
void bp_points_destroy(bp_points *set);
size_t bp_points_count(const bp_points *set);
/* n_msm MSMs of `terms` terms each over the first `terms` points of the set; MSM j takes scalars[j*terms .. (j+1)*terms).
 * Device form: d_scalars / d_outs (n_msm x 32 B) / d_status (n_msm bytes, optional) are device pointers, nothing is synchronised.
 * Host form: pinned memory recommended; synchronises. */
int bp_msm_points_device(bp_ctx *ctx, bp_points *set, const void *d_scalars, size_t n_msm, size_t terms, void *d_outs, void *d_status);
int bp_msm_points(bp_ctx *ctx, bp_points *set, const uint8_t *scalars, size_t n_msm, size_t terms, uint8_t *outs, uint8_t *status);

/* ---- inner-product prover, device-resident (no generator folding) ---------------------------- */
/* InnerProductProof::create (src/inner_product_proof.rs:38-193) for n_proofs proofs of the same length N side by side.  The vectors
 * a, b, G_factors, H_factors stay on the device; the points are never folded -- round j's L and R are MSMs of N + 1 terms over the
 * ORIGINAL generators with the accumulated challenge products as coefficients (same group elements, hence the same proof bytes, as
 * the reference's folded form :127-134,177-178) -- so a round is O(N) scalar products and one MSM launch chain for all proofs.
 * The host keeps the transcripts: round() returns L, R (:87-113,153-163), the caller appends them, draws u (:118-121,168-171) and
 * calls fold(u, u^-1) (:122-134,172-178); after lg N rounds finish() returns the final a, b (:187-192).
 *   begin        : G, H = BulletproofGens::G(n, m) / H(n, m) of the resident table, N = n*m
 *   begin_points : arbitrary G, H (N compressed points each)
 *   Q  : n_proofs x 32 B;  a, b : n_proofs x N canonical scalars;  G_factors / H_factors : likewise, or NULL for all ones. */
typedef struct bp_ippx bp_ippx;
int bp_ippx_begin(bp_ctx *ctx, bp_gens *gens, size_t n, size_t m, size_t n_proofs, const uint8_t *Q, const uint8_t *G_factors, const uint8_t *H_factors,
                  const uint8_t *a, const uint8_t *b, bp_ippx **out);
int bp_ippx_begin_points(bp_ctx *ctx, const uint8_t *G, const uint8_t *H, size_t N, size_t n_proofs, const uint8_t *Q, const uint8_t *G_factors, const uint8_t *H_factors,
                         const uint8_t *a, const uint8_t *b, bp_ippx **out);
size_t bp_ippx_current_len(const bp_ippx *sess);
int bp_ippx_round(bp_ippx *sess, uint8_t *LR_out /* n_proofs x 64 */);
int bp_ippx_fold(bp_ippx *sess, const uint8_t *u /* n_proofs x 32 */, const uint8_t *u_inv);
int bp_ippx_finish(bp_ippx *sess, uint8_t *ab_out /* n_proofs x 64 */);
void bp_ippx_end(bp_ippx *sess);

/* ---- generator tables ---------------------------------------------------------------------- */
/* BulletproofGens::new(gens_capacity, party_capacity) + PedersenGens::default()
 * (generators.rs:44-53,157-204): SHAKE256 expansion on the host, Elligator maps and the
 * table (affine Niels form, 96 B/point) on the device, where it stays resident. */
int bp_gens_create(bp_ctx *ctx, size_t gens_capacity, size_t party_capacity, bp_gens **out);
void bp_gens_destroy(bp_gens *gens);
/* compressed generator: which = 0 -> G, 1 -> H (party, index); 2 -> B; 3 -> B_blinding */
int bp_gens_get(bp_gens *gens, int which, size_t party, size_t index, uint8_t out[32]);
/* device pointer + size of the resident table, layout [B_blinding, B, G[party][i]..., H[party][i]...]:
 * this is the buffer broadcast once over NCCL at start-up (SURVEY.md §8e). */
int bp_gens_device_table(bp_gens *gens, void **d_table, size_t *bytes);
/* an uninitialised table of the same geometry, to be filled by a broadcast from rank 0 */
int bp_gens_create_empty(bp_ctx *ctx, size_t gens_capacity, size_t party_capacity, bp_gens **out);

/* ---- range proofs -------------------------------------------------------------------------- */
/* Batch verifier (SURVEY.md §8a row A6): `count` proofs with the same (n, m), each proof_len =
 * 32*(9 + 2*lg(n*m)) bytes as written by RangeProof::to_bytes (range_proof/mod.rs:487-499), each
 * with m commitments.  Every proof is checked exactly as RangeProof::verify_multiple
 * (range_proof/mod.rs:345-452) would: verdict[i] = BP_PROOF_OK iff the reference returns Ok(()).
 * All proofs start from the same transcript state.  Internally one random-linear-combination
 * MSM covers the whole batch; if it does not vanish, every proof is re-checked on its own.
 * seed: 32 bytes of external randomness for the batching weights, or NULL to draw from the OS.  The weights of a proof
 * (the reference's `c = Scalar::random(rng)`, mod.rs:396, and the proof's weight in the combination) are squeezed from a fork
 * of that proof's final transcript state keyed with the seed -- merlin's `build_rng().finalize(rng)` construction -- so they are
 * bound to the proof bytes even when the caller's seed is fixed or known. */
int bp_rangeproof_verify_batch(bp_ctx *ctx, bp_gens *gens, const uint8_t transcript[BP_TRANSCRIPT_BYTES],
                               const uint8_t *proofs, size_t proof_len, const uint8_t *commitments,
                               size_t n, size_t m, size_t count, const uint8_t seed[32], uint8_t *verdicts);
/* Asynchronous form for pipelining host buffers (pinned memory recommended): queues the H2D copies,
 * all kernels and the D2H copy of the verdicts on the context's stream; call
 * bp_rangeproof_verify_finish() to synchronise and run the rare per-proof fallback. */
int bp_rangeproof_verify_begin(bp_ctx *ctx, bp_gens *gens, const uint8_t transcript[BP_TRANSCRIPT_BYTES],
                               const uint8_t *proofs, size_t proof_len, const uint8_t *commitments,
                               size_t n, size_t m, size_t count, const uint8_t seed[32]);
int bp_rangeproof_verify_finish(bp_ctx *ctx, uint8_t *verdicts);
/* Device-resident form: proofs/commitments are device pointers; verdicts stay on the device
 * (count x uint32) and nothing is synchronised, so calls can be queued back to back on one context.
 * There is no per-proof recheck on this path: if the combined check fails, every well-formed proof of the
 * batch is marked BP_PROOF_VERIFICATION_ERROR and *h_batch_ok_pinned (optional, pinned) becomes 0 — rerun such a
 * batch through bp_rangeproof_verify_batch for per-proof verdicts.  Used for the HBM-resident throughput measurement. */
int bp_rangeproof_verify_batch_device(bp_ctx *ctx, bp_gens *gens, const uint8_t transcript[BP_TRANSCRIPT_BYTES],
                                      const void *d_proofs, size_t proof_len, const void *d_commitments,
                                      size_t n, size_t m, size_t count, const uint8_t seed[32], void *d_verdicts_u32,
                                      uint32_t *h_batch_ok_pinned);

/* Launch groups: `n_batches` (<= 256) independent batches of `count` proofs each in ONE launch sequence.  Every batch keeps its own
 * random-linear-combination MSM, its own accept flag and its own per-proof fallback; only the kernel launches are shared, so that
 * the grids of a group fill the 148 SMs where a single 1024-proof batch gives most kernels less than one wave.
 * proofs / commitments / verdicts are laid out batch after batch (n_batches*count entries); batch_ok (optional): n_batches flags,
 * 1 = every proof of that batch accepted.  The single-batch entry points above are the n_batches = 1 case. */
int bp_rangeproof_verify_group_begin(bp_ctx *ctx, bp_gens *gens, const uint8_t transcript[BP_TRANSCRIPT_BYTES],
                                     const uint8_t *proofs, size_t proof_len, const uint8_t *commitments,
                                     size_t n, size_t m, size_t count, size_t n_batches, const uint8_t seed[32]);
int bp_rangeproof_verify_group_finish(bp_ctx *ctx, uint8_t *verdicts, uint8_t *batch_ok);
/* Between *_begin and *_finish the context's arenas belong to the pending verification (its reject path reads them): every other
 * entry point on that context returns BP_ERR_INVALID_ARGUMENT with a message in bp_last_error(); use another context for concurrent work.
 * A failed *_begin leaves nothing pending. */
/* device-resident form (see bp_rangeproof_verify_batch_device); h_batch_ok_pinned (optional, pinned): n_batches x uint32 */
int bp_rangeproof_verify_group_device(bp_ctx *ctx, bp_gens *gens, const uint8_t transcript[BP_TRANSCRIPT_BYTES],
                                      const void *d_proofs, size_t proof_len, const void *d_commitments,
                                      size_t n, size_t m, size_t count, size_t n_batches, const uint8_t seed[32], void *d_verdicts_u32,
                                      uint32_t *h_batch_ok_pinned);
/* Reserve a geometry on a context: sizes every arena the verification of n_batches x count (n, m)-proofs touches, builds the
 * term->point maps, captures the launch sequence as a CUDA graph (two branches: decompression beside transcript replay) and runs
 * it once.  Afterwards no call with this geometry allocates, and each call costs one parameter upload + one graph launch.
 * Other geometries still work on the same context (direct launches, arenas grown on demand). */
int bp_rangeproof_verify_reserve(bp_ctx *ctx, bp_gens *gens, size_t n, size_t m, size_t count, size_t n_batches);

/* D2D copy of the resident table to / from a caller-owned device buffer of bp_gens_device_table() bytes
 * (the Python harness broadcasts a torch tensor with NCCL and imports it on the other ranks). */
int bp_gens_table_export(bp_gens *gens, void *d_dst);
int bp_gens_table_import(bp_gens *gens, const void *d_src);

/* ---- per-kernel timing (CUDA events on the launching stream; used by bench.py's roofline block) ---- */
int bp_prof_enable(bp_ctx *ctx, int on);
int bp_prof_kernel_count(void);
const char *bp_prof_kernel_name(int kernel_id);
int bp_prof_report(bp_ctx *ctx, double *ms, uint64_t *counts);
/* Per-launch records (kernel id, start, end in ms relative to the first record of `ref`, another context of the same device)
 * accumulated since profiling was enabled; does not clear them.  Diagnostic for multi-stream overlap (benchmarks/timeline.py). */
int bp_prof_timeline(bp_ctx *ctx, bp_ctx *ref, int *kernel_ids, double *start_ms, double *end_ms, size_t cap, size_t *n_out);

/* ---- host helpers -------------------------------------------------------------------------- */
/* merlin::Transcript for callers without the Rust crate (same framing as transcript.rs:43-94 expects):
 * Transcript::new(label), append_message, append_u64, challenge_bytes on the 203-byte wire state. */
void bp_transcript_new(const uint8_t *label, size_t len, uint8_t out[BP_TRANSCRIPT_BYTES]);
void bp_transcript_append_message(uint8_t state[BP_TRANSCRIPT_BYTES], const char *label, const uint8_t *msg, size_t len);
void bp_transcript_append_u64(uint8_t state[BP_TRANSCRIPT_BYTES], const char *label, uint64_t x);
void bp_transcript_challenge_bytes(uint8_t state[BP_TRANSCRIPT_BYTES], const char *label, uint8_t *out, size_t len);

/* ---- test hook ----------------------------------------------------------------------------- */
/* element-wise field operation on the device over n pairs of 32-byte little-endian values:
 * op 0 add, 1 sub, 2 mul, 3 invert(a), 4 a^((p-5)/8), 5 neg(a), 6 a^2, 7 (a+b)(a-b); canonical bytes out */
int bp_debug_fe_op(bp_ctx *ctx, int op, const uint8_t *a, const uint8_t *b, size_t n, uint8_t *out);

#ifdef __cplusplus
}
#endif
#endif
