// C ABI of the engine (include/bpmsm.h): context, scratch arenas, kernel orchestration.
// No CPU fallback: every entry point needs a usable CUDA device and fails with BP_ERR_CUDA otherwise.
#include <cuda_runtime.h>
#include <sys/random.h>
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <array>
#include <cstring>
#include <memory>
#include <string>
#include <type_traits>
#include <vector>
#include "../../include/bpmsm.h"
#include "../../include/bpmsm_ct.h"
#include "kernels.cuh"

static_assert(BP_TRANSCRIPT_BYTES == 203, "transcript wire size");

namespace {

// Owned allocation: device memory (cudaMalloc) or pinned host memory (cudaMallocHost), freed by the destructor.  Non-copyable, so a
// handle or arena can be released only by its owner.  ensure() grows scratch with headroom; alloc() sizes a fixed array exactly.
template <bool Pinned> struct Buf {
    void *p = nullptr; size_t cap = 0;
    Buf() = default;
    Buf(const Buf &) = delete;
    Buf &operator=(const Buf &) = delete;
    ~Buf() { release(); }
    cudaError_t ensure(size_t bytes) { return bytes <= cap ? cudaSuccess : alloc(bytes + bytes / 4 + 256); }
    cudaError_t alloc(size_t bytes) {
        release();
        cudaError_t e = Pinned ? cudaMallocHost(&p, bytes) : cudaMalloc(&p, bytes);
        if (e == cudaSuccess) cap = bytes; else p = nullptr;
        return e;
    }
    void release() {
        if (p) { if (Pinned) cudaFreeHost(p); else cudaFree(p); }
        p = nullptr; cap = 0;
    }
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};
using DevBuf = Buf<false>;
using HostBuf = Buf<true>;

enum KernelId { KID_DECOMPRESS, KID_COMPRESS, KID_FROM_UNIFORM, KID_MSM_COUNT, KID_MSM_SCAN, KID_MSM_SCATTER, KID_MSM_ACCUMULATE, KID_MSM_REDUCE,
                KID_MSM_COMBINE, KID_RP_TRANSCRIPT, KID_RP_HEAD, KID_RP_SCALARS, KID_RP_DECOMPRESS, KID_RP_STATIC_REDUCE, KID_IPP_FOLD, KID_SMALL,
                KID_MSM_CT_RECODE, KID_MSM_CT_TABLE, KID_MSM_CT_STRAUS, KID_MSM_CT_REDUCE, KID_COUNT };
const char *const KERNEL_NAMES[KID_COUNT] = {"k_decompress", "k_compress", "k_from_uniform", "k_msm_count", "k_msm_scan", "k_msm_scatter", "k_msm_accumulate",
                                             "k_msm_reduce", "k_msm_combine", "k_rp_transcript", "k_rp_head", "k_rp_scalars", "k_rp_decompress", "k_rp_static_reduce", "k_ipp_fold", "small_kernels",
                                             "k_msm_ct_recode", "k_msm_ct_table", "k_msm_ct_straus", "k_msm_ct_reduce"};
struct ProfRec { int kid; cudaEvent_t a, b; };

struct VerifyState {          // what bp_rangeproof_verify_*begin leaves for *_finish
    bool active = false; rp_geom g{}; uint32_t total = 0, n_batches = 1; bp_gens *gens = nullptr; uint8_t param_verdict = 0;
};
struct MsmArena { DevBuf counts, starts, cursor, order, sorted, buckets, wsums; };      // scratch of one Pippenger pipeline pass
struct MsmPlan { int c = 0, W = 0; uint32_t nb = 0, heavy_min = 0; size_t segs = 0, n_buckets = 0, heavy_cap = 0; uint32_t n_msm = 0, T = 0; };

// Everything whose address the verifier's launch graph bakes in (rp_chain's kernel arguments).  Private to the verifier: no other entry
// point can regrow -- i.e. move -- one of these buffers.  Holds DevBufs only, so signature() walks it as an array and a buffer added
// here is covered without further bookkeeping.
struct RpGraphScratch {
    DevBuf par, contrib, part, scalars, status, decbad, niels, pidx, offsets, results, batch_ok, combined, chal, tabs, raw, pow2_tab;
    MsmArena ar;
    uint64_t signature() const {         // FNV-1a over the addresses: a regrown (moved) buffer invalidates the graph
        const DevBuf *b = reinterpret_cast<const DevBuf *>(this);
        uint64_t h = 1469598103934665603ULL;
        for (size_t i = 0; i < sizeof *this / sizeof(DevBuf); i++) { h ^= (uint64_t)(uintptr_t)b[i].p; h *= 1099511628211ULL; }
        return h;
    }
};
static_assert(std::is_standard_layout<RpGraphScratch>::value && sizeof(RpGraphScratch) % sizeof(DevBuf) == 0, "RpGraphScratch holds DevBufs only");

}  // namespace

#define BP_MAX_GROUP_BATCHES 256

struct bp_ctx {
    int device = 0, sm_count = 148; cudaStream_t stream = nullptr; bool own_stream = false;
    cudaStream_t aux = nullptr; cudaEvent_t ev_fork = nullptr, ev_join = nullptr;    // second branch of the verifier's launch graph
    std::string err; uint64_t launches = 0;
    int msm_window = 0;                                       // 0 = by size (msm_pick_window); bp_ctx_set_msm_window pins it (tuning / tests)
    bool prof_on = false; std::vector<ProfRec> prof;          // per-kernel CUDA-event timing (bp_prof_*)
    // MSM scratch
    DevBuf in_scalars, in_points, in_offsets, niels, ok, msm_err, results, outs, flags, ix_pidx;
    MsmArena ar_gen;          // bp_msm*, indexed MSMs, IPP rounds, the verifier's per-proof fallback
    DevBuf ct_digits, ct_tab, ct_chunks, ct_part;                  // constant-time indexed MSM: digits, [1..8]P tables, chunk bounds, chunk partials
    // range-proof scratch.  The inputs and verdicts stay outside rp: the kernels read their addresses from the parameter block
    // (rp.par), not from graph arguments, so they may move without invalidating the graph.
    RpGraphScratch rp;
    DevBuf rp_proofs, rp_commit, rp_verdict;
    DevBuf fb_scalars, fb_pidx, fb_offsets;
    HostBuf h_verdict;                                               // pinned
    HostBuf h_flag;                                                  // pinned: combined_ok[BP_MAX_GROUP_BATCHES] | batch_ok[BP_MAX_GROUP_BATCHES]
    // pinned staging ring for the per-call parameter block of the verifier: a slot is reused only after the upload queued from it has
    // completed, so back-to-back device-path calls on one context never see each other's parameters
    static const int STAGE_SLOTS = 8;
    HostBuf h_stage; cudaEvent_t stage_ev[STAGE_SLOTS] = {}; unsigned stage_next = 0;
    VerifyState vs;
    size_t pidx_key[6] = {0, 0, 0, 0, 0, 0};                        // geometry the cached rp.pidx / rp.offsets were built for
    // reserved geometry: every arena sized, launch sequence captured as a CUDA graph
    cudaGraphExec_t graph = nullptr; std::array<size_t, 6> graph_key{}; uint64_t graph_launches = 0, graph_sig = 0;
    ~bp_ctx() {
        if (graph) cudaGraphExecDestroy(graph);
        for (cudaEvent_t e : stage_ev) if (e) cudaEventDestroy(e);
        if (ev_fork) cudaEventDestroy(ev_fork);
        if (ev_join) cudaEventDestroy(ev_join);
        if (aux) cudaStreamDestroy(aux);
        if (own_stream) cudaStreamDestroy(stream);
    }
};

struct bp_gens {
    bp_ctx *ctx = nullptr; size_t cap = 0, parties = 0, n_points = 0;
    DevBuf table;                      // n_points entries: [B_blinding, B, G[party][i].., H[party][i]..]
    ge_niels *d_table() const { return table.as<ge_niels>(); }
};

struct bp_points {
    bp_ctx *ctx = nullptr; size_t n = 0;
    DevBuf pts, idx;                   // n decompressed points; term -> point map of idx_T terms (k_iota_mod over idx_len)
    size_t idx_T = 0, idx_len = 0;
};

struct bp_ipp {
    bp_ctx *ctx = nullptr; uint32_t N = 0;
    DevBuf pts;                        // [G (N) | H (N) | Q]
    DevBuf scal, idx, offs;
};

struct bp_ippx {
    bp_ctx *ctx = nullptr; uint32_t N = 0, B = 0, n = 0;
    const ge_niels *d_static = nullptr; DevBuf own_pts;                   // the gens table, or the session's own [G (N) | H (N)]
    DevBuf d_q;                                                           // B points Q
    DevBuf a, b, cG, cH, gidx, hidx, scal, pidx, offs, in, outs;
};

namespace {

#define CK(ctx, call)                                                                                  \
    do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { (ctx)->err = std::string(#call) + ": " + cudaGetErrorString(e_); return BP_ERR_CUDA; } } while (0)
#define LAUNCH_CHECK(ctx)                                                                              \
    do { (ctx)->launches++; cudaError_t e_ = cudaGetLastError(); if (e_ != cudaSuccess) { (ctx)->err = std::string("kernel launch: ") + cudaGetErrorString(e_); return BP_ERR_CUDA; } } while (0)

// launch wrapper: counts the launch and, when profiling is enabled, brackets it with CUDA events on the launching stream
#define LAUNCH(ctx, kid, ...)                                                                          \
    do {                                                                                               \
        ProfRec pr_{(kid), nullptr, nullptr};                                                          \
        if ((ctx)->prof_on) { cudaEventCreate(&pr_.a); cudaEventCreate(&pr_.b); cudaEventRecord(pr_.a, (ctx)->stream); } \
        __VA_ARGS__;                                                                                   \
        if ((ctx)->prof_on) { cudaEventRecord(pr_.b, (ctx)->stream); (ctx)->prof.push_back(pr_); }     \
        LAUNCH_CHECK(ctx);                                                                             \
    } while (0)

// the fallback of a pending begin/finish verification reads the context's scratch arenas: other entry points must not run in between
#define BUSY_CHECK(c) do { if ((c)->vs.active) { (c)->err = "a range-proof verification is pending on this context: call bp_rangeproof_verify_group_finish first"; return BP_ERR_INVALID_ARGUMENT; } } while (0)

inline unsigned blocks_for(size_t n, unsigned threads) { return (unsigned)((n + threads - 1) / threads); }

// ---------------------------------------------------------------- host Keccak (SHAKE256 / SHA3-512) for the generator chain
struct HostSponge {
    uint64_t st[25]; unsigned rate, pos; uint8_t pad; bool squeezing;
    HostSponge(unsigned r, uint8_t p) : rate(r), pos(0), pad(p), squeezing(false) { memset(st, 0, sizeof st); }
    void xor_byte(unsigned i, uint8_t b) { st[i >> 3] ^= (uint64_t)b << (8 * (i & 7)); }
    uint8_t get_byte(unsigned i) const { return (uint8_t)(st[i >> 3] >> (8 * (i & 7))); }
    void absorb(const uint8_t *d, size_t n) { for (size_t i = 0; i < n; i++) { xor_byte(pos++, d[i]); if (pos == rate) { keccak_f1600(st); pos = 0; } } }
    void squeeze(uint8_t *o, size_t n) {
        if (!squeezing) { xor_byte(pos, pad); xor_byte(rate - 1, 0x80); keccak_f1600(st); pos = 0; squeezing = true; }
        for (size_t i = 0; i < n; i++) { if (pos == rate) { keccak_f1600(st); pos = 0; } o[i] = get_byte(pos++); }
    }
};

// ---------------------------------------------------------------- the Pippenger pipeline
struct MsmArgs {
    const uint8_t *d_scalars; const uint32_t *d_offsets; uint32_t n_msm, T;
    const uint32_t *d_point_idx; const ge_niels *d_static, *d_dynamic; uint32_t *d_err; int window;
};

MsmPlan msm_make_plan(uint32_t T, uint32_t n_msm, int window) {
    MsmPlan p; p.T = T; p.n_msm = n_msm;
    size_t avg = ((size_t)T + n_msm - 1) / n_msm;
    p.c = window > 0 ? window : msm_pick_window(avg);
    p.W = msm_num_windows(p.c);
    p.nb = 1u << (p.c - 1);
    p.segs = (size_t)n_msm * p.W; p.n_buckets = p.segs * p.nb;
    // heavy-bucket threshold: far above the mean bucket size, and large enough that a block per bucket pays off.
    // A bucket holds >= heavy_min entries, so at most T*W/heavy_min of them exist.
    p.heavy_min = (uint32_t)std::max<size_t>(256, 8 * (avg / p.nb + 1));
    p.heavy_cap = std::min<size_t>(p.n_buckets, (size_t)T * p.W / p.heavy_min + 1);
    return p;
}
// arenas of one pipeline pass (grow-only; no CUDA call when they are already large enough, which is what lets a reserved
// geometry run under stream capture)
int msm_ensure(bp_ctx *ctx, MsmArena &ar, const MsmPlan &p) {
    // counts | size histogram | bin cursors share one allocation so a single memset clears them
    CK(ctx, ar.counts.ensure((p.n_buckets + 2 * MSM_SIZE_BINS + 4) * 4)); CK(ctx, ar.starts.ensure(p.n_buckets * 4)); CK(ctx, ar.cursor.ensure(p.n_buckets * 4));
    CK(ctx, ar.order.ensure((p.n_buckets + p.heavy_cap) * 4));
    CK(ctx, ar.sorted.ensure((size_t)p.T * p.W * 4)); CK(ctx, ar.buckets.ensure(p.n_buckets * sizeof(ge_ext))); CK(ctx, ar.wsums.ensure(p.segs * sizeof(ge_ext)));
    return BP_OK;
}
int msm_launch(bp_ctx *ctx, MsmArena &ar, const MsmArgs &a, const MsmPlan &p, ge_ext *d_results) {
    const int c = p.c, W = p.W; const uint32_t nb = p.nb, heavy_min = p.heavy_min; const size_t segs = p.segs, n_buckets = p.n_buckets;
    uint32_t *size_hist = ar.counts.as<uint32_t>() + n_buckets, *bin_cursor = size_hist + MSM_SIZE_BINS, *heavy_n = bin_cursor + MSM_SIZE_BINS;
    uint32_t *heavy = ar.order.as<uint32_t>() + n_buckets;
    cudaStream_t s = ctx->stream;
    CK(ctx, cudaMemsetAsync(ar.counts.p, 0, (n_buckets + 2 * MSM_SIZE_BINS + 4) * 4, s));
    LAUNCH(ctx, KID_MSM_COUNT, k_msm_count<<<blocks_for(a.T, 256), 256, 0, s>>>(a.d_scalars, a.d_offsets, a.n_msm, a.T, c, W, ar.counts.as<uint32_t>(), a.d_err));
    LAUNCH(ctx, KID_MSM_SCAN, k_msm_scan<<<(unsigned)segs, 256, 0, s>>>(ar.counts.as<uint32_t>(), nb, ar.starts.as<uint32_t>(), ar.cursor.as<uint32_t>(), size_hist));
    LAUNCH(ctx, KID_MSM_SCAN, k_msm_order<<<blocks_for(n_buckets, 256), 256, 0, s>>>(ar.counts.as<uint32_t>(), n_buckets, size_hist, bin_cursor, ar.order.as<uint32_t>(), heavy_min, heavy_n, heavy));
    LAUNCH(ctx, KID_MSM_SCATTER, k_msm_scatter<<<blocks_for(a.T, 256), 256, 0, s>>>(a.d_scalars, a.d_offsets, a.n_msm, a.T, c, W, ar.cursor.as<uint32_t>(), ar.sorted.as<uint32_t>()));
    // two lanes per bucket once buckets hold >= 8 terms on average: half the serial chain per thread and twice the warps in flight for
    // one extra addition per bucket (config 2: 108 -> 71 us alone, same throughput with 24 batches in flight; profiles/r1_timeline.md)
    size_t avg = ((size_t)a.T + a.n_msm - 1) / a.n_msm;
    const int acc_split = avg / nb >= 8 && n_buckets < 65536 ? 2 : 1;
    const unsigned heavy_blocks = (unsigned)std::min<size_t>(p.heavy_cap, 148);
#define ACC_LAUNCH(SP) do { unsigned light_ = blocks_for(n_buckets * SP, MSM_ACC_THREADS); \
        LAUNCH(ctx, KID_MSM_ACCUMULATE, k_msm_accumulate<SP><<<light_ + heavy_blocks, MSM_ACC_THREADS, 0, s>>>(ar.starts.as<uint32_t>(), ar.cursor.as<uint32_t>(), ar.sorted.as<uint32_t>(), \
        a.d_offsets, ar.order.as<uint32_t>(), W, nb, n_buckets, a.d_point_idx, a.d_static, a.d_dynamic, ar.buckets.as<ge_ext>(), heavy_min, light_, heavy_n, heavy)); } while (0)
    if (acc_split == 2) ACC_LAUNCH(2); else ACC_LAUNCH(1);
#undef ACC_LAUNCH
    // two warps per segment up to 2048 buckets (fewer scan / tree additions per useful bucket addition); eight for the wide windows of
    // large MSMs, where a segment's 16k-32k buckets would otherwise be 256-512 sequential additions per thread
    unsigned rthreads = nb >= 4096 ? 256 : nb >= 64 ? 64 : 32;
    LAUNCH(ctx, KID_MSM_REDUCE, k_msm_reduce<<<(unsigned)segs, rthreads, 0, s>>>(ar.buckets.as<ge_ext>(), nb, ar.wsums.as<ge_ext>()));
    if (a.n_msm <= 256)      // few MSMs: the Horner chain is pure latency -> four cooperating lanes per MSM
        LAUNCH(ctx, KID_MSM_COMBINE, k_msm_combine4<<<blocks_for(a.n_msm, 8), 32, 0, s>>>(ar.wsums.as<ge_ext>(), a.n_msm, c, W, d_results));
    else
        LAUNCH(ctx, KID_MSM_COMBINE, k_msm_combine<<<blocks_for(a.n_msm, 32), 32, 0, s>>>(ar.wsums.as<ge_ext>(), a.n_msm, c, W, d_results));
    return BP_OK;
}
int msm_core(bp_ctx *ctx, const MsmArgs &a, ge_ext *d_results) {       // generic arena
    if (a.T == 0) return BP_ERR_INVALID_ARGUMENT;
    MsmPlan p = msm_make_plan(a.T, a.n_msm, a.window > 0 ? a.window : ctx->msm_window);
    int rc = msm_ensure(ctx, ctx->ar_gen, p);
    if (rc) return rc;
    return msm_launch(ctx, ctx->ar_gen, a, p, d_results);
}

__global__ void k_mark_invalid(const uint8_t *ok, const uint32_t *offsets, uint32_t n_msm, uint32_t T, uint32_t *msm_err) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T || ok[t]) return;
    atomicOr(msm_err + (n_msm == 1 ? 0u : msm_of_term(offsets, n_msm, t)), 1u);
}
__global__ void k_msm_status(const uint32_t *msm_err, uint32_t n_msm, uint8_t *status) {
    uint32_t m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n_msm) return;
    uint32_t e = msm_err[m];
    status[m] = (e & 2u) ? BP_ERR_NONCANONICAL_SCALAR : (e & 1u) ? BP_ERR_INVALID_POINT : BP_OK;
}
__global__ void k_rp_point_idx(rp_geom g, uint32_t gens_cap, uint32_t gens_parties, uint32_t count, int per_proof_rows, uint32_t dyn_base, uint32_t *out) {
    // combined layout, per batch: [S static | count*D dynamic] (g.nbatch batches);  per-proof rows: count x [S static | D dynamic].
    // Dynamic indices address the decompressed per-proof points: (first proof of the batch + q)*D + d, plus dyn_base.
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t total = per_proof_rows ? (size_t)count * (g.S + g.D) : (size_t)g.nbatch * g.T;
    if (i >= total) return;
    uint32_t t, dyn;
    if (per_proof_rows) { uint32_t p = (uint32_t)(i / (g.S + g.D)); t = (uint32_t)(i % (g.S + g.D)); dyn = dyn_base + p * g.D + (t - g.S); }
    else { uint32_t b = (uint32_t)(i / g.T); t = (uint32_t)(i % g.T); dyn = dyn_base + b * g.count * g.D + (t - g.S); if (t > g.S) t = g.S; }
    uint32_t v;
    if (t < 2) v = t;                                                                       // B_blinding, B
    else if (t < 2 + g.N) { uint32_t q = t - 2; v = gens_slot(0u, q / g.n, q % g.n, gens_cap, gens_parties); }
    else if (t < g.S) { uint32_t q = t - 2 - g.N; v = gens_slot(1u, q / g.n, q % g.n, gens_cap, gens_parties); }
    else v = BP_POINT_DYNAMIC | dyn;
    out[i] = v;
}
// decompress to the four extended coordinates (X, Y, Z = 1, T), 4 x 32 canonical bytes per point: the in-memory RistrettoPoint
// a host caller keeps (bp_decompress_batch / bp_compress_batch)
__global__ void __launch_bounds__(128) k_decompress_xyzt(const uint8_t *__restrict__ in, size_t n, uint8_t *__restrict__ out, uint8_t *__restrict__ ok) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t s[32]; ld32(s, in + 32 * i);
    fe x, y; bool valid = ge_decode(x, y, s);
    if (!valid) { x = fe_zero(); y = fe_one(); }
    uint8_t b[32];
    fe_tobytes(b, x); st32(out + 128 * i, b); fe_tobytes(b, y); st32(out + 128 * i + 32, b);
    fe_tobytes(b, fe_one()); st32(out + 128 * i + 64, b); fe_tobytes(b, fe_mul(x, y)); st32(out + 128 * i + 96, b);
    ok[i] = valid ? 1 : 0;
}
__global__ void __launch_bounds__(128) k_compress_xyzt(const uint8_t *__restrict__ in, size_t n, uint8_t *__restrict__ out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ge_ext p; uint8_t b[32];
    ld32(b, in + 128 * i); p.X = fe_frombytes_raw(b); ld32(b, in + 128 * i + 32); p.Y = fe_frombytes_raw(b);
    ld32(b, in + 128 * i + 64); p.Z = fe_frombytes_raw(b); ld32(b, in + 128 * i + 96); p.T = fe_frombytes_raw(b);
    uint8_t s[32]; ge_encode(s, p); st32(out + 32 * i, s);
}
// term -> point map of n_msm equal-length MSMs over the same resident point set: term t uses point t mod len
__global__ void k_iota_mod(uint32_t T, uint32_t len, uint32_t *out) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < T) out[t] = t % len;
}
__global__ void k_fill_offsets(uint32_t n, uint32_t stride, uint32_t *out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= n) out[i] = i * stride;
}

// ---------------------------------------------------------------- steps shared by the entry points
// decompress n points that must all be valid (resident point sets, IPP generators and Q); synchronises
int decompress_checked(bp_ctx *c, const uint8_t *d_compressed, size_t n, ge_niels *out) {
    CK(c, c->ok.ensure(n));
    LAUNCH(c, KID_DECOMPRESS, k_decompress<<<blocks_for(n, 128), 128, 0, c->stream>>>(d_compressed, n, out, c->ok.as<uint8_t>()));
    std::vector<uint8_t> ok(n);
    CK(c, cudaMemcpyAsync(ok.data(), c->ok.p, n, cudaMemcpyDeviceToHost, c->stream)); CK(c, cudaStreamSynchronize(c->stream));
    for (uint8_t v : ok) if (!v) return BP_ERR_INVALID_POINT;
    return BP_OK;
}
// the MSMs of `a` on the generic arena, compressed to d_outs (a.n_msm x 32 B); with d_status, a.d_err turned into status codes
int msm_to_bytes(bp_ctx *c, const MsmArgs &a, uint8_t *d_outs, uint8_t *d_status) {
    int rc = msm_core(c, a, c->results.as<ge_ext>());
    if (rc) return rc;
    LAUNCH(c, KID_COMPRESS, k_compress<<<blocks_for(a.n_msm, 128), 128, 0, c->stream>>>(c->results.as<ge_ext>(), a.n_msm, d_outs));
    if (d_status) { LAUNCH(c, KID_SMALL, k_msm_status<<<blocks_for(a.n_msm, 128), 128, 0, c->stream>>>(a.d_err, a.n_msm, d_status)); }
    return BP_OK;
}
// host-buffer forms: the results and status codes the device form left in c->outs / c->flags back to the caller; synchronises
int msm_copy_out(bp_ctx *c, size_t n_msm, uint8_t *outs, uint8_t *status) {
    std::vector<uint8_t> st(n_msm);
    CK(c, cudaMemcpyAsync(outs, c->outs.p, n_msm * 32, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaMemcpyAsync(st.data(), c->flags.p, n_msm, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    if (status) memcpy(status, st.data(), n_msm);
    return BP_OK;
}

// ---------------------------------------------------------------- handle construction: a handle reaches the caller only once complete
int points_from_device(bp_ctx *c, const uint8_t *d_compressed, size_t n, bp_points **out) {
    std::unique_ptr<bp_points> h(new bp_points()); h->ctx = c; h->n = n;
    CK(c, h->pts.alloc(n * sizeof(ge_niels)));
    int rc = decompress_checked(c, d_compressed, n, h->pts.as<ge_niels>());
    if (rc) return rc;
    *out = h.release(); return BP_OK;
}
// the table is allocated at exactly n_points entries: no headroom on what may be the largest allocation of the process
int gens_alloc(bp_ctx *c, size_t cap, size_t parties, std::unique_ptr<bp_gens> &g) {
    if (!c || cap == 0 || parties == 0) return BP_ERR_INVALID_ARGUMENT;
    CK(c, cudaSetDevice(c->device));
    g.reset(new bp_gens());
    g->ctx = c; g->cap = cap; g->parties = parties; g->n_points = 2 + 2 * cap * parties;
    CK(c, g->table.alloc(g->n_points * sizeof(ge_niels)));
    return BP_OK;
}
int ippx_alloc(bp_ctx *c, size_t N, size_t B, std::unique_ptr<bp_ippx> &s) {
    if (!c || N == 0 || (N & (N - 1)) || B == 0 || 2 * B * (N + 1) >= (1u << 31)) return BP_ERR_INVALID_ARGUMENT;      // power of two (inner_product_proof.rs:67)
    BUSY_CHECK(c);
    CK(c, cudaSetDevice(c->device));
    s.reset(new bp_ippx()); s->ctx = c; s->N = (uint32_t)N; s->B = (uint32_t)B; s->n = (uint32_t)N;
    size_t BN = B * N;
    CK(c, s->d_q.alloc(B * sizeof(ge_niels)));
    for (DevBuf *b : {&s->a, &s->b, &s->cG, &s->cH}) CK(c, b->ensure(BN * sizeof(sc)));
    CK(c, s->gidx.ensure(N * 4)); CK(c, s->hidx.ensure(N * 4)); CK(c, s->scal.ensure(2 * B * (N + 1) * 32)); CK(c, s->pidx.ensure(2 * B * (N + 1) * 4));
    CK(c, s->offs.ensure((2 * B + 1) * 4)); CK(c, s->in.ensure(std::max<size_t>(4 * BN * 32, 64 * B))); CK(c, s->outs.ensure(64 * B));
    return BP_OK;
}
int check_scalars_canonical(const uint8_t *s, size_t n) {
    for (size_t i = 0; i < n; i++) if (sc_geq_l(sc_load(s + 32 * i))) return BP_ERR_NONCANONICAL_SCALAR;
    return BP_OK;
}
// common tail of the two begin forms: Q points, scalar vectors (B x N canonical scalars each; Gf / Hf may be NULL = all ones)
int ippx_load(bp_ippx *s, const uint8_t *Q, const uint8_t *Gf, const uint8_t *Hf, const uint8_t *a, const uint8_t *b) {
    bp_ctx *c = s->ctx; cudaStream_t st = c->stream; size_t BN = (size_t)s->B * s->N;
    for (const uint8_t *v : {a, b}) if (check_scalars_canonical(v, BN)) return BP_ERR_NONCANONICAL_SCALAR;
    for (const uint8_t *v : {Gf, Hf}) if (v && check_scalars_canonical(v, BN)) return BP_ERR_NONCANONICAL_SCALAR;
    uint8_t *din = s->in.as<uint8_t>();
    CK(c, cudaMemcpyAsync(din, a, BN * 32, cudaMemcpyHostToDevice, st)); CK(c, cudaMemcpyAsync(din + BN * 32, b, BN * 32, cudaMemcpyHostToDevice, st));
    if (Gf) CK(c, cudaMemcpyAsync(din + 2 * BN * 32, Gf, BN * 32, cudaMemcpyHostToDevice, st));
    if (Hf) CK(c, cudaMemcpyAsync(din + 3 * BN * 32, Hf, BN * 32, cudaMemcpyHostToDevice, st));
    ippx_geom g{s->N, s->B, s->n};
    LAUNCH(c, KID_SMALL, k_ippx_init<<<blocks_for(BN, 128), 128, 0, st>>>(g, din, din + BN * 32, Gf ? din + 2 * BN * 32 : nullptr, Hf ? din + 3 * BN * 32 : nullptr,
                                                                         s->a.as<sc>(), s->b.as<sc>(), s->cG.as<sc>(), s->cH.as<sc>()));
    CK(c, c->in_points.ensure((size_t)s->B * 32));
    CK(c, cudaMemcpyAsync(c->in_points.p, Q, (size_t)s->B * 32, cudaMemcpyHostToDevice, st));
    int rc = decompress_checked(c, c->in_points.as<uint8_t>(), s->B, s->d_q.as<ge_niels>());
    if (rc) return rc;
    LAUNCH(c, KID_SMALL, k_fill_offsets<<<blocks_for((size_t)2 * s->B + 1, 256), 256, 0, st>>>(2 * s->B, s->N + 1, s->offs.as<uint32_t>()));
    return BP_OK;
}

// ---------------------------------------------------------------- range proofs
// Parameter checks of verify_multiple_with_rng (mod.rs:358-366) and of from_bytes / verification_scalars
// that depend only on (proof_len, n, m): one verdict for the whole call, or BP_PROOF_OK to go on.
uint8_t rp_param_verdict(const bp_gens *gens, size_t proof_len, size_t n, size_t m, rp_geom *g) {
    if (proof_len % 32 != 0 || proof_len < 7 * 32) return BP_PROOF_FORMAT_ERROR;                 // mod.rs:498-503
    size_t ne = (proof_len - 7 * 32) / 32;
    if (ne < 2 || (ne - 2) % 2 != 0 || (ne - 2) / 2 >= 32) return BP_PROOF_FORMAT_ERROR;         // inner_product_proof.rs:375-388
    size_t k = (ne - 2) / 2;
    if (!(n == 8 || n == 16 || n == 32 || n == 64)) return BP_PROOF_INVALID_BITSIZE;
    if (gens->cap < n || gens->parties < m) return BP_PROOF_INVALID_GENERATORS_LENGTH;
    if (m == 0 || n * m != ((size_t)1 << k) || k > BP_MAX_LG_N) return BP_PROOF_VERIFICATION_ERROR;   // inner_product_proof.rs:204-211
    g->n = (uint32_t)n; g->m = (uint32_t)m; g->k = (uint32_t)k; g->N = (uint32_t)(n * m);
    g->D = (uint32_t)(4 + 2 * k + m); g->S = 2 + 2 * g->N; g->proof_len = (uint32_t)proof_len;
    return BP_PROOF_OK;
}
bool rp_set_group(rp_geom *g, size_t count, size_t n_batches) {
    if (count == 0 || n_batches == 0 || n_batches > BP_MAX_GROUP_BATCHES || count >= (1u << 24)) return false;
    size_t T = (size_t)g->S + count * g->D;
    if (T * n_batches >= (1u << 31) || count * n_batches >= (1u << 24)) return false;
    g->count = (uint32_t)count; g->nbatch = (uint32_t)n_batches; g->T = (uint32_t)T;
    return true;
}

// every arena of one launch group (grow-only); after this nothing on the verification path allocates
int rp_ensure(bp_ctx *c, const rp_geom &g) {
    size_t total = (size_t)g.count * g.nbatch, TT = (size_t)g.T * g.nbatch;
    RpGraphScratch &r = c->rp;
    CK(c, r.par.ensure(sizeof(rp_params)));
    CK(c, r.contrib.ensure(total * g.S * sizeof(sc))); CK(c, r.scalars.ensure(TT * 32));
    CK(c, r.part.ensure((size_t)g.nbatch * ((g.count + RP_CHUNK - 1) / RP_CHUNK) * g.S * sizeof(sc)));
    CK(c, r.status.ensure(total * 4)); CK(c, r.decbad.ensure(total * 4)); CK(c, r.niels.ensure(total * g.D * sizeof(ge_niels)));
    CK(c, r.pidx.ensure(TT * 4)); CK(c, r.offsets.ensure(((size_t)g.nbatch + 1) * 4)); CK(c, r.results.ensure((size_t)g.nbatch * sizeof(ge_ext)));
    CK(c, r.batch_ok.ensure((size_t)g.nbatch * 4)); CK(c, r.combined.ensure((size_t)g.nbatch * 4));
    CK(c, r.chal.ensure(total * sizeof(rp_head))); CK(c, r.tabs.ensure(total * rp_tab_size(g.k, g.m) * sizeof(sc)));
    CK(c, r.raw.ensure(total * (RP_RAW_U + g.k) * 64));
    if (c->h_verdict.cap < total * 4) CK(c, c->h_verdict.alloc(total * 4));
    if (!r.pow2_tab.p) {             // 2^e (e < 64) in Montgomery form, computed once per context with the host build of sc.cuh
        std::vector<sc> tab(64);
        for (int e = 0; e < 64; e++) tab[e] = sc_mont_from_u64(1ULL << e);
        CK(c, r.pow2_tab.ensure(64 * sizeof(sc)));
        CK(c, cudaMemcpyAsync(r.pow2_tab.p, tab.data(), 64 * sizeof(sc), cudaMemcpyHostToDevice, c->stream)); CK(c, cudaStreamSynchronize(c->stream));
    }
    return msm_ensure(c, r.ar, msm_make_plan((uint32_t)TT, g.nbatch, 0));
}
// what a captured graph was built for besides the scratch addresses: the geometry and the table address (a kernel argument of the captured nodes)
std::array<size_t, 6> rp_graph_key(const bp_gens *gens, const rp_geom &g) { return {g.n, g.m, g.count, g.nbatch, (size_t)(uintptr_t)gens->table.p, g.proof_len}; }
// term -> point map and MSM offsets of the combined MSMs: depend only on the geometry, rebuilt when it changes
int rp_build_maps(bp_ctx *c, bp_gens *gens, const rp_geom &g) {
    size_t key[6] = {g.n, g.m, g.count, g.nbatch, gens->cap, gens->parties};
    if (memcmp(key, c->pidx_key, sizeof key) == 0) return BP_OK;
    cudaStream_t s = c->stream;
    LAUNCH(c, KID_SMALL, k_rp_point_idx<<<blocks_for((size_t)g.T * g.nbatch, 256), 256, 0, s>>>(g, (uint32_t)gens->cap, (uint32_t)gens->parties, g.count, 0, 0, c->rp.pidx.as<uint32_t>()));
    LAUNCH(c, KID_SMALL, k_fill_offsets<<<blocks_for((size_t)g.nbatch + 1, 256), 256, 0, s>>>(g.nbatch, g.T, c->rp.offsets.as<uint32_t>()));
    memcpy(c->pidx_key, key, sizeof key);
    return BP_OK;
}
// upload the per-call parameter block through the pinned staging ring, so that the asynchronous upload never reads caller
// memory after the entry point returns
int rp_upload_params(bp_ctx *c, const uint8_t *h_transcript, const uint8_t *seed, const uint8_t *d_proofs, const uint8_t *d_commit, uint32_t *d_verdict) {
    unsigned slot = c->stage_next++ % bp_ctx::STAGE_SLOTS;
    CK(c, cudaEventSynchronize(c->stage_ev[slot]));                          // the upload that last used this slot is done
    rp_params *par = reinterpret_cast<rp_params *>(c->h_stage.as<uint8_t>() + 512 * slot);
    memset(par, 0, sizeof *par);
    memcpy(par->tstate, h_transcript, BP_TRANSCRIPT_BYTES);
    if (seed) memcpy(par->seed, seed, 32);
    else if (getrandom(par->seed, 32, 0) != 32) { c->err = "getrandom failed"; return BP_ERR_CUDA; }
    par->proofs = d_proofs; par->commitments = d_commit; par->verdict = d_verdict;
    CK(c, cudaMemcpyAsync(c->rp.par.p, par, sizeof *par, cudaMemcpyHostToDevice, c->stream));
    CK(c, cudaEventRecord(c->stage_ev[slot], c->stream));
    return BP_OK;
}

// The launch sequence of one group, launches only (no allocation, no synchronisation: capturable).  Two branches: the
// decompressions need nothing but the proof bytes and run beside the transcript replay and the head.
int rp_chain(bp_ctx *c, bp_gens *gens, const rp_geom &g) {
    cudaStream_t s = c->stream, s2 = c->prof_on ? c->stream : c->aux;
    const uint32_t total = g.count * g.nbatch;
    RpGraphScratch &r = c->rp;
    const rp_params *par = r.par.as<rp_params>();
    uint8_t *d_scal = r.scalars.as<uint8_t>();
    if (s2 != s) { CK(c, cudaEventRecord(c->ev_fork, s)); CK(c, cudaStreamWaitEvent(s2, c->ev_fork, 0)); }
    CK(c, cudaMemsetAsync(r.decbad.p, 0, (size_t)total * 4, s2));
    const size_t dec_smem = (size_t)(RP_DEC_THREADS / g.D + 2) * (g.proof_len + 32 * g.m);
    LAUNCH(c, KID_RP_DECOMPRESS, k_rp_decompress<<<blocks_for((size_t)total * g.D, RP_DEC_THREADS), RP_DEC_THREADS, dec_smem, s2>>>(par, g, total, r.niels.as<ge_niels>(), r.decbad.as<uint32_t>()));
    if (s2 != s) CK(c, cudaEventRecord(c->ev_join, s2));
    LAUNCH(c, KID_RP_TRANSCRIPT, k_rp_transcript<<<blocks_for(total, RP_TR_THREADS), RP_TR_THREADS, 0, s>>>(par, g, total, r.raw.as<uint8_t>(), r.status.as<uint32_t>()));
    LAUNCH(c, KID_RP_HEAD, k_rp_head_seq<<<blocks_for(total, 32), 32, 0, s>>>(par, g, r.raw.as<uint8_t>(), total, r.chal.as<rp_head>(), r.tabs.as<sc>(),
                                                                                  r.pow2_tab.as<sc>(), r.status.as<uint32_t>()));
    if (s2 != s) CK(c, cudaStreamWaitEvent(s, c->ev_join, 0));
    const uint32_t nchunks = (g.count + RP_CHUNK - 1) / RP_CHUNK;
    LAUNCH(c, KID_RP_SCALARS, k_rp_scalars_sum<<<g.nbatch * nchunks, (unsigned)std::min<uint32_t>(128, std::max<uint32_t>(32, g.N)), 0, s>>>(g, r.chal.as<rp_head>(), r.tabs.as<sc>(),
                                                                                  r.decbad.as<uint32_t>(), r.part.as<sc>(), d_scal));
    LAUNCH(c, KID_RP_STATIC_REDUCE, k_rp_static_sum<<<dim3(g.S, g.nbatch), 32, 0, s>>>(r.part.as<sc>(), g, d_scal));
    MsmArgs a{d_scal, r.offsets.as<uint32_t>(), g.nbatch, g.T * g.nbatch, r.pidx.as<uint32_t>(), gens->d_table(), r.niels.as<ge_niels>(), nullptr, 0};
    int rc = msm_launch(c, r.ar, a, msm_make_plan(a.T, a.n_msm, 0), r.results.as<ge_ext>());
    if (rc) return rc;
    LAUNCH(c, KID_SMALL, k_rp_verdict_batch<<<g.nbatch, 256, 0, s>>>(r.status.as<uint32_t>(), r.decbad.as<uint32_t>(), r.results.as<ge_ext>(), g, par,
                                                                      r.batch_ok.as<uint32_t>(), r.combined.as<uint32_t>()));
    return BP_OK;
}

bool rp_graph_matches(const bp_ctx *c, const bp_gens *gens, const rp_geom &g) {
    return c->graph && rp_graph_key(gens, g) == c->graph_key && c->graph_sig == c->rp.signature();
}
// queue everything up to the verdicts; d_proofs / d_commitments are device pointers
int rp_verify_queue(bp_ctx *c, bp_gens *gens, const rp_geom &g, const uint8_t *d_proofs, const uint8_t *d_commit,
                    const uint8_t *h_transcript, const uint8_t *seed, uint32_t *d_verdict) {
    const bool use_graph = !c->prof_on && rp_graph_matches(c, gens, g);
    if (!use_graph) { int rc = rp_ensure(c, g); if (rc) return rc; }
    int rc = rp_build_maps(c, gens, g);          // another geometry may have used the context since: the maps follow the key
    if (rc) return rc;
    rc = rp_upload_params(c, h_transcript, seed, d_proofs, d_commit, d_verdict);
    if (rc) return rc;
    if (use_graph) { CK(c, cudaGraphLaunch(c->graph, c->stream)); c->launches += c->graph_launches; return BP_OK; }
    return rp_chain(c, gens, g);
}

// per-proof re-check of the proofs [p0, p0 + count) of a group: count independent MSMs of S + D terms
int rp_fallback_range(bp_ctx *c, bp_gens *gens, const rp_geom &g, uint32_t p0, uint32_t count, uint32_t *d_verdict) {
    cudaStream_t s = c->stream;
    uint32_t row = g.S + g.D; size_t T = (size_t)count * row;
    if (T >= (1u << 31)) { c->err = "fallback batch too large"; return BP_ERR_INVALID_ARGUMENT; }
    CK(c, c->fb_scalars.ensure(T * 32)); CK(c, c->fb_pidx.ensure(T * 4)); CK(c, c->fb_offsets.ensure(((size_t)count + 1) * 4));
    CK(c, c->results.ensure((size_t)count * sizeof(ge_ext)));
    uint32_t batch = p0 / g.count, q0 = p0 % g.count;
    const uint8_t *dyn = c->rp.scalars.as<uint8_t>() + ((size_t)batch * g.T + g.S + (size_t)q0 * g.D) * 32;
    LAUNCH(c, KID_SMALL, k_rp_expand_scalars<<<blocks_for(T, 128), 128, 0, s>>>(c->rp.contrib.as<sc>() + (size_t)p0 * g.S, dyn, g, count, c->fb_scalars.as<uint8_t>()));
    LAUNCH(c, KID_SMALL, k_rp_point_idx<<<blocks_for(T, 256), 256, 0, s>>>(g, (uint32_t)gens->cap, (uint32_t)gens->parties, count, 1, p0 * g.D, c->fb_pidx.as<uint32_t>()));
    LAUNCH(c, KID_SMALL, k_fill_offsets<<<blocks_for((size_t)count + 1, 256), 256, 0, s>>>(count, row, c->fb_offsets.as<uint32_t>()));
    MsmArgs a{c->fb_scalars.as<uint8_t>(), c->fb_offsets.as<uint32_t>(), count, (uint32_t)T, c->fb_pidx.as<uint32_t>(), gens->d_table(), c->rp.niels.as<ge_niels>(), nullptr, 0};
    int rc = msm_core(c, a, c->results.as<ge_ext>());
    if (rc) return rc;
    LAUNCH(c, KID_SMALL, k_rp_verdict_proofs<<<blocks_for(count, 128), 128, 0, s>>>(c->rp.status.as<uint32_t>() + p0, c->rp.decbad.as<uint32_t>() + p0, c->results.as<ge_ext>(), count, d_verdict + p0));
    return BP_OK;
}
// A batch whose combined check failed.  Level 1: one combined MSM per chunk of RP_CHUNK proofs, from the partial sums the main path
// already holds (one pipeline pass over the batch's ~T terms).  Level 2: the proofs of the failing chunks, each with its own MSM
// (mod.rs:421-447 per proof).  One bad proof in 1024 costs two small passes instead of 1024 147-term MSMs.
int rp_verify_fallback(bp_ctx *c, bp_gens *gens, const rp_geom &g, uint32_t batch, uint32_t *d_verdict, bool *contrib_ready) {
    cudaStream_t s = c->stream;
    const uint32_t nch = (g.count + RP_CHUNK - 1) / RP_CHUNK, row = g.S + RP_CHUNK * g.D, p0 = batch * g.count;
    size_t T = (size_t)nch * row;
    if (T >= (1u << 31)) { c->err = "fallback batch too large"; return BP_ERR_INVALID_ARGUMENT; }
    CK(c, c->fb_scalars.ensure(T * 32)); CK(c, c->fb_pidx.ensure(T * 4)); CK(c, c->fb_offsets.ensure(((size_t)nch + 1) * 4));
    CK(c, c->results.ensure((size_t)nch * sizeof(ge_ext))); CK(c, c->flags.ensure((size_t)nch * 4));
    LAUNCH(c, KID_SMALL, k_rp_chunk_rows<<<blocks_for(T, 128), 128, 0, s>>>(c->rp.part.as<sc>() + (size_t)batch * nch * g.S, c->rp.scalars.as<uint8_t>() + ((size_t)batch * g.T + g.S) * 32, g,
                                                                              (uint32_t)gens->cap, (uint32_t)gens->parties, p0 * g.D, c->fb_scalars.as<uint8_t>(), c->fb_pidx.as<uint32_t>()));
    LAUNCH(c, KID_SMALL, k_fill_offsets<<<blocks_for((size_t)nch + 1, 256), 256, 0, s>>>(nch, row, c->fb_offsets.as<uint32_t>()));
    MsmArgs a{c->fb_scalars.as<uint8_t>(), c->fb_offsets.as<uint32_t>(), nch, (uint32_t)T, c->fb_pidx.as<uint32_t>(), gens->d_table(), c->rp.niels.as<ge_niels>(), nullptr, 0};
    int rc = msm_core(c, a, c->results.as<ge_ext>());
    if (rc) return rc;
    LAUNCH(c, KID_SMALL, k_rp_verdict_chunks<<<blocks_for(g.count, 128), 128, 0, s>>>(c->rp.status.as<uint32_t>() + p0, c->rp.decbad.as<uint32_t>() + p0, c->results.as<ge_ext>(), g.count,
                                                                                      d_verdict + p0, c->flags.as<uint32_t>()));
    std::vector<uint32_t> ok(nch);
    CK(c, cudaMemcpyAsync(ok.data(), c->flags.p, (size_t)nch * 4, cudaMemcpyDeviceToHost, s)); CK(c, cudaStreamSynchronize(s));
    uint32_t nfail = 0; for (uint32_t v : ok) nfail += v ? 0 : 1;
    if (nfail == 0) return BP_OK;       // cannot happen when the batch's combination failed, short of a 2^-128 cancellation between chunk weights
    if (!*contrib_ready) {   // the combined path keeps only sums: the per-proof static-term scalars are produced here, on the reject path (whole group; idempotent)
        const uint32_t total = g.count * g.nbatch;
        LAUNCH(c, KID_RP_SCALARS, k_rp_scalars<<<blocks_for((size_t)total * (g.N + g.D), 128), 128, 0, s>>>(g, c->rp.chal.as<rp_head>(), c->rp.tabs.as<sc>(), c->rp.decbad.as<uint32_t>(), total,
                                                                                                            c->rp.contrib.as<sc>(), c->rp.scalars.as<uint8_t>()));
        *contrib_ready = true;
    }
    if (nfail > 4) return rp_fallback_range(c, gens, g, p0, g.count, d_verdict);      // many bad chunks: one pass over the whole batch
    for (uint32_t ch = 0; ch < nch; ch++)
        if (!ok[ch]) { rc = rp_fallback_range(c, gens, g, p0 + ch * RP_CHUNK, std::min<uint32_t>(RP_CHUNK, g.count - ch * RP_CHUNK), d_verdict); if (rc) return rc; }
    return BP_OK;
}

}  // namespace

// ================================================================================================ C ABI
extern "C" {

int bp_ctx_create(int device, void *stream, bp_ctx **out) {
    if (!out) return BP_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return BP_ERR_CUDA;
    if (cudaSetDevice(device) != cudaSuccess) return BP_ERR_CUDA;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major < 10) return BP_ERR_CUDA;   // sm_100a only
    std::unique_ptr<bp_ctx> c(new bp_ctx());
    c->device = device; c->sm_count = prop.multiProcessorCount > 0 ? prop.multiProcessorCount : 148;
    if (stream) { c->stream = (cudaStream_t)stream; c->own_stream = false; }
    else { if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) return BP_ERR_CUDA; c->own_stream = true; }
    if (c->h_flag.alloc(2 * BP_MAX_GROUP_BATCHES * 4) != cudaSuccess || c->h_stage.alloc(512 * bp_ctx::STAGE_SLOTS) != cudaSuccess) return BP_ERR_CUDA;
    for (cudaEvent_t &e : c->stage_ev) if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return BP_ERR_CUDA;
    if (cudaStreamCreateWithFlags(&c->aux, cudaStreamNonBlocking) != cudaSuccess) return BP_ERR_CUDA;
    // k_rp_decompress stages the proofs its block touches in dynamic shared memory: up to 13 proofs of 32*(9+2*20) + 32*m bytes
    if (cudaFuncSetAttribute(k_rp_decompress, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024) != cudaSuccess) return BP_ERR_CUDA;
    if (cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming) != cudaSuccess || cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming) != cudaSuccess) return BP_ERR_CUDA;
    *out = c.release();
    return BP_OK;
}
void bp_ctx_destroy(bp_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    if (c->aux) cudaStreamSynchronize(c->aux);
    delete c;
}
const char *bp_last_error(const bp_ctx *c) { return c ? c->err.c_str() : "null context"; }
uint64_t bp_ctx_launch_count(const bp_ctx *c) { return c ? c->launches : 0; }
int bp_ctx_set_msm_window(bp_ctx *c, int window_bits) { if (!c || window_bits < 0 || window_bits > 18 || window_bits == 1) return BP_ERR_INVALID_ARGUMENT; c->msm_window = window_bits; return BP_OK; }
int bp_ctx_synchronize(bp_ctx *c) { if (!c) return BP_ERR_INVALID_ARGUMENT; CK(c, cudaSetDevice(c->device)); CK(c, cudaStreamSynchronize(c->stream)); return BP_OK; }

int bp_decompress_check_batch(bp_ctx *c, const uint8_t *points, size_t n, uint8_t *ok) {
    if (!c || !points || !ok) return BP_ERR_INVALID_ARGUMENT;
    BUSY_CHECK(c);
    if (n == 0) return BP_OK;
    CK(c, cudaSetDevice(c->device));
    CK(c, c->in_points.ensure(n * 32)); CK(c, c->niels.ensure(n * sizeof(ge_niels))); CK(c, c->ok.ensure(n));
    CK(c, cudaMemcpyAsync(c->in_points.p, points, n * 32, cudaMemcpyHostToDevice, c->stream));
    LAUNCH(c, KID_DECOMPRESS, k_decompress<<<blocks_for(n, 128), 128, 0, c->stream>>>(c->in_points.as<uint8_t>(), n, c->niels.as<ge_niels>(), c->ok.as<uint8_t>()));
    CK(c, cudaMemcpyAsync(ok, c->ok.p, n, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return BP_OK;
}

int bp_from_uniform_bytes_batch(bp_ctx *c, const uint8_t *uniform, size_t n, uint8_t *points_out) {
    if (!c || !uniform || !points_out) return BP_ERR_INVALID_ARGUMENT;
    BUSY_CHECK(c);
    if (n == 0) return BP_OK;
    CK(c, cudaSetDevice(c->device));
    CK(c, c->in_points.ensure(n * 64)); CK(c, c->outs.ensure(n * 32));
    CK(c, cudaMemcpyAsync(c->in_points.p, uniform, n * 64, cudaMemcpyHostToDevice, c->stream));
    LAUNCH(c, KID_FROM_UNIFORM, k_from_uniform<<<blocks_for(n, 128), 128, 0, c->stream>>>(c->in_points.as<uint8_t>(), n, nullptr, c->outs.as<uint8_t>()));
    CK(c, cudaMemcpyAsync(points_out, c->outs.p, n * 32, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return BP_OK;
}

int bp_msm_batch_device(bp_ctx *c, const void *d_scalars, const void *d_points, const void *d_offsets_u32, size_t n_msm, size_t total_terms,
                        void *d_outs, void *d_status) {
    if (!c || !d_scalars || !d_points || !d_offsets_u32 || !d_outs || n_msm == 0) return BP_ERR_INVALID_ARGUMENT;
    if (total_terms == 0 || total_terms >= (1u << 31) || n_msm >= (1u << 31)) return BP_ERR_INVALID_ARGUMENT;
    BUSY_CHECK(c);
    CK(c, cudaSetDevice(c->device));
    uint32_t T = (uint32_t)total_terms, M = (uint32_t)n_msm;
    CK(c, c->niels.ensure((size_t)T * sizeof(ge_niels))); CK(c, c->ok.ensure(T)); CK(c, c->msm_err.ensure((size_t)M * 4)); CK(c, c->results.ensure((size_t)M * sizeof(ge_ext)));
    cudaStream_t s = c->stream;
    CK(c, cudaMemsetAsync(c->msm_err.p, 0, (size_t)M * 4, s));
    LAUNCH(c, KID_DECOMPRESS, k_decompress<<<blocks_for(T, 128), 128, 0, s>>>((const uint8_t *)d_points, T, c->niels.as<ge_niels>(), c->ok.as<uint8_t>()));
    LAUNCH(c, KID_SMALL, k_mark_invalid<<<blocks_for(T, 256), 256, 0, s>>>(c->ok.as<uint8_t>(), (const uint32_t *)d_offsets_u32, M, T, c->msm_err.as<uint32_t>()));
    MsmArgs a{(const uint8_t *)d_scalars, (const uint32_t *)d_offsets_u32, M, T, nullptr, nullptr, c->niels.as<ge_niels>(), c->msm_err.as<uint32_t>(), 0};
    return msm_to_bytes(c, a, (uint8_t *)d_outs, (uint8_t *)d_status);
}

int bp_msm_batch(bp_ctx *c, const uint8_t *scalars, const uint8_t *points, const uint64_t *offsets, size_t n_msm, uint8_t *outs, uint8_t *status) {
    if (!c || !offsets || !outs || n_msm == 0) return BP_ERR_INVALID_ARGUMENT;
    size_t T = offsets[n_msm];
    if (offsets[0] != 0 || T >= (1u << 31)) return BP_ERR_INVALID_ARGUMENT;
    for (size_t j = 0; j < n_msm; j++) if (offsets[j + 1] < offsets[j]) return BP_ERR_LENGTH_MISMATCH;
    CK(c, cudaSetDevice(c->device));
    if (T == 0) {                      // every MSM empty: the identity encodes as 32 zero bytes
        memset(outs, 0, 32 * n_msm); if (status) memset(status, 0, n_msm); return BP_OK;
    }
    if (!scalars || !points) return BP_ERR_INVALID_ARGUMENT;
    std::vector<uint32_t> off32(n_msm + 1);
    for (size_t j = 0; j <= n_msm; j++) off32[j] = (uint32_t)offsets[j];
    CK(c, c->in_scalars.ensure(T * 32)); CK(c, c->in_points.ensure(T * 32)); CK(c, c->in_offsets.ensure((n_msm + 1) * 4));
    CK(c, c->outs.ensure(n_msm * 32)); CK(c, c->flags.ensure(n_msm));
    cudaStream_t s = c->stream;
    CK(c, cudaMemcpyAsync(c->in_scalars.p, scalars, T * 32, cudaMemcpyHostToDevice, s));
    CK(c, cudaMemcpyAsync(c->in_points.p, points, T * 32, cudaMemcpyHostToDevice, s));
    CK(c, cudaMemcpyAsync(c->in_offsets.p, off32.data(), (n_msm + 1) * 4, cudaMemcpyHostToDevice, s));
    int rc = bp_msm_batch_device(c, c->in_scalars.p, c->in_points.p, c->in_offsets.p, n_msm, T, c->outs.p, c->flags.p);
    if (rc) return rc;
    return msm_copy_out(c, n_msm, outs, status);
}

int bp_msm(bp_ctx *c, const uint8_t *scalars, const uint8_t *points, size_t n, uint8_t out[32]) {
    uint64_t off[2] = {0, n}; uint8_t st = 0;
    int rc = bp_msm_batch(c, scalars, points, off, 1, out, &st);
    return rc ? rc : st;
}

// ---------------------------------------------------------------------------------------------- point values across the boundary
int bp_decompress_batch(bp_ctx *c, const uint8_t *points, size_t n, uint8_t *xyzt_out, uint8_t *ok) {
    if (!c || !points || !xyzt_out || !ok) return BP_ERR_INVALID_ARGUMENT;
    if (n == 0) return BP_OK;
    BUSY_CHECK(c);
    CK(c, cudaSetDevice(c->device));
    CK(c, c->in_points.ensure(n * 32)); CK(c, c->outs.ensure(n * 128)); CK(c, c->ok.ensure(n));
    CK(c, cudaMemcpyAsync(c->in_points.p, points, n * 32, cudaMemcpyHostToDevice, c->stream));
    LAUNCH(c, KID_DECOMPRESS, k_decompress_xyzt<<<blocks_for(n, 128), 128, 0, c->stream>>>(c->in_points.as<uint8_t>(), n, c->outs.as<uint8_t>(), c->ok.as<uint8_t>()));
    CK(c, cudaMemcpyAsync(xyzt_out, c->outs.p, n * 128, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaMemcpyAsync(ok, c->ok.p, n, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return BP_OK;
}
int bp_compress_batch(bp_ctx *c, const uint8_t *xyzt, size_t n, uint8_t *points_out) {
    if (!c || !xyzt || !points_out) return BP_ERR_INVALID_ARGUMENT;
    if (n == 0) return BP_OK;
    BUSY_CHECK(c);
    CK(c, cudaSetDevice(c->device));
    CK(c, c->in_points.ensure(n * 128)); CK(c, c->outs.ensure(n * 32));
    CK(c, cudaMemcpyAsync(c->in_points.p, xyzt, n * 128, cudaMemcpyHostToDevice, c->stream));
    LAUNCH(c, KID_COMPRESS, k_compress_xyzt<<<blocks_for(n, 128), 128, 0, c->stream>>>(c->in_points.as<uint8_t>(), n, c->outs.as<uint8_t>()));
    CK(c, cudaMemcpyAsync(points_out, c->outs.p, n * 32, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return BP_OK;
}

// ---------------------------------------------------------------------------------------------- resident point sets (decompressed once, reused by many MSMs)
int bp_points_create(bp_ctx *c, const uint8_t *points, size_t n, bp_points **out) {
    if (!out) return BP_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    if (!c || !points || n == 0 || n >= (1u << 31)) return BP_ERR_INVALID_ARGUMENT;
    BUSY_CHECK(c);
    CK(c, cudaSetDevice(c->device));
    CK(c, c->in_points.ensure(n * 32));
    CK(c, cudaMemcpyAsync(c->in_points.p, points, n * 32, cudaMemcpyHostToDevice, c->stream));
    return points_from_device(c, c->in_points.as<uint8_t>(), n, out);
}
int bp_points_create_device(bp_ctx *c, const void *d_points, size_t n, bp_points **out) {
    if (!out) return BP_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    if (!c || !d_points || n == 0 || n >= (1u << 31)) return BP_ERR_INVALID_ARGUMENT;
    BUSY_CHECK(c);
    CK(c, cudaSetDevice(c->device));
    return points_from_device(c, (const uint8_t *)d_points, n, out);
}
void bp_points_destroy(bp_points *h) { if (!h) return; cudaSetDevice(h->ctx->device); cudaStreamSynchronize(h->ctx->stream); delete h; }
size_t bp_points_count(const bp_points *h) { return h ? h->n : 0; }

// n_msm MSMs of `terms` terms each over the first `terms` points of the set (MSM j uses scalars[j*terms .. (j+1)*terms)); device pointers,
// nothing synchronised.  No decompression on this path: 32 B of scalar per term is all that is read from the caller.
int bp_msm_points_device(bp_ctx *c, bp_points *h, const void *d_scalars, size_t n_msm, size_t terms, void *d_outs, void *d_status) {
    if (!c || !h || !d_scalars || !d_outs || n_msm == 0 || terms == 0 || terms > h->n || n_msm * terms >= (1u << 31)) return BP_ERR_INVALID_ARGUMENT;
    BUSY_CHECK(c);
    CK(c, cudaSetDevice(c->device));
    uint32_t T = (uint32_t)(n_msm * terms), M = (uint32_t)n_msm;
    cudaStream_t s = c->stream;
    if (h->idx_T < T || h->idx_len != terms) {
        CK(c, cudaStreamSynchronize(s));
        h->idx_T = 0;
        CK(c, h->idx.alloc((size_t)T * 4));
        LAUNCH(c, KID_SMALL, k_iota_mod<<<blocks_for(T, 256), 256, 0, s>>>(T, (uint32_t)terms, h->idx.as<uint32_t>()));
        h->idx_T = T; h->idx_len = terms;
    }
    CK(c, c->in_offsets.ensure(((size_t)M + 1) * 4)); CK(c, c->msm_err.ensure((size_t)M * 4)); CK(c, c->results.ensure((size_t)M * sizeof(ge_ext)));
    LAUNCH(c, KID_SMALL, k_fill_offsets<<<blocks_for((size_t)M + 1, 256), 256, 0, s>>>(M, (uint32_t)terms, c->in_offsets.as<uint32_t>()));
    CK(c, cudaMemsetAsync(c->msm_err.p, 0, (size_t)M * 4, s));
    MsmArgs a{(const uint8_t *)d_scalars, c->in_offsets.as<uint32_t>(), M, T, h->idx.as<uint32_t>(), h->pts.as<ge_niels>(), nullptr, c->msm_err.as<uint32_t>(), 0};
    return msm_to_bytes(c, a, (uint8_t *)d_outs, (uint8_t *)d_status);
}
// host-buffer form (pinned memory recommended): H2D of the scalars, the MSMs, D2H of the 32-byte results; synchronises
int bp_msm_points(bp_ctx *c, bp_points *h, const uint8_t *scalars, size_t n_msm, size_t terms, uint8_t *outs, uint8_t *status) {
    if (!c || !h || !scalars || !outs || n_msm == 0 || terms == 0) return BP_ERR_INVALID_ARGUMENT;
    BUSY_CHECK(c);
    CK(c, cudaSetDevice(c->device));
    size_t T = n_msm * terms;
    CK(c, c->in_scalars.ensure(T * 32)); CK(c, c->outs.ensure(n_msm * 32)); CK(c, c->flags.ensure(n_msm));
    CK(c, cudaMemcpyAsync(c->in_scalars.p, scalars, T * 32, cudaMemcpyHostToDevice, c->stream));
    int rc = bp_msm_points_device(c, h, c->in_scalars.p, n_msm, terms, c->outs.p, c->flags.p);
    if (rc) return rc;
    return msm_copy_out(c, n_msm, outs, status);
}

// ---------------------------------------------------------------------------------------------- generators
int bp_gens_create_empty(bp_ctx *c, size_t cap, size_t parties, bp_gens **out) {
    if (!out) return BP_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    std::unique_ptr<bp_gens> g;
    int rc = gens_alloc(c, cap, parties, g);
    if (rc) return rc;
    *out = g.release();
    return BP_OK;
}

int bp_gens_create(bp_ctx *c, size_t cap, size_t parties, bp_gens **out) {
    if (!out) return BP_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    std::unique_ptr<bp_gens> g;
    int rc = gens_alloc(c, cap, parties, g);
    if (rc) return rc;
    // ristretto255 basepoint, compressed (RISTRETTO_BASEPOINT_COMPRESSED)
    static const uint8_t BASEPOINT[32] = {0xe2, 0xf2, 0xae, 0x0a, 0x6a, 0xbc, 0x4e, 0x71, 0xa8, 0x84, 0xa9, 0x61, 0xc5, 0x00, 0x51, 0x5f,
                                          0x58, 0xe3, 0x0b, 0x6a, 0xa5, 0x82, 0xdd, 0x8d, 0xb6, 0xa6, 0x59, 0x45, 0xe0, 0x8d, 0x2d, 0x76};
    // uniform bytes: slot 0 = SHA3-512(B) for B_blinding (generators.rs:48-51); slot 1 unused (B is decompressed);
    // then the SHAKE256("GeneratorsChain" || tag || LE32(party)) streams (generators.rs:62-104,179-204)
    std::vector<uint8_t> uni(g->n_points * 64, 0);
    { HostSponge h(72, 0x06); h.absorb(BASEPOINT, 32); h.squeeze(uni.data(), 64); }
    for (int which = 0; which < 2; which++)
        for (size_t p = 0; p < parties; p++) {
            HostSponge h(136, 0x1f);
            uint8_t label[5] = {(uint8_t)(which ? 'H' : 'G'), (uint8_t)p, (uint8_t)(p >> 8), (uint8_t)(p >> 16), (uint8_t)(p >> 24)};
            h.absorb((const uint8_t *)"GeneratorsChain", 15); h.absorb(label, 5);
            h.squeeze(uni.data() + 64 * (2 + (which * parties + p) * cap), 64 * cap);
        }
    CK(c, c->in_points.ensure(uni.size())); CK(c, c->in_scalars.ensure(32));
    cudaStream_t s = c->stream;
    CK(c, cudaMemcpyAsync(c->in_points.p, uni.data(), uni.size(), cudaMemcpyHostToDevice, s));
    CK(c, cudaMemcpyAsync(c->in_scalars.p, BASEPOINT, 32, cudaMemcpyHostToDevice, s));
    LAUNCH(c, KID_FROM_UNIFORM, k_from_uniform<<<blocks_for(g->n_points, 128), 128, 0, s>>>(c->in_points.as<uint8_t>(), g->n_points, g->d_table(), nullptr));
    LAUNCH(c, KID_DECOMPRESS, k_decompress<<<1, 128, 0, s>>>(c->in_scalars.as<uint8_t>(), 1, g->d_table() + 1, nullptr));
    CK(c, cudaStreamSynchronize(s));
    *out = g.release();
    return BP_OK;
}
void bp_gens_destroy(bp_gens *g) { if (!g) return; cudaSetDevice(g->ctx->device); delete g; }
int bp_gens_device_table(bp_gens *g, void **d_table, size_t *bytes) {
    if (!g || !d_table || !bytes) return BP_ERR_INVALID_ARGUMENT;
    *d_table = g->table.p; *bytes = g->n_points * sizeof(ge_niels); return BP_OK;
}
int bp_gens_get(bp_gens *g, int which, size_t party, size_t index, uint8_t out[32]) {
    if (!g || !out) return BP_ERR_INVALID_ARGUMENT;
    bp_ctx *c = g->ctx; size_t slot;
    if (which == 2) slot = 1; else if (which == 3) slot = 0;
    else if ((which == 0 || which == 1) && party < g->parties && index < g->cap) slot = gens_slot<size_t>(which, party, index, g->cap, g->parties);
    else return BP_ERR_INVALID_ARGUMENT;
    CK(c, cudaSetDevice(c->device)); CK(c, c->outs.ensure(32));
    LAUNCH(c, KID_SMALL, k_niels_to_compressed<<<1, 32, 0, c->stream>>>(g->d_table() + slot, 1, c->outs.as<uint8_t>()));
    CK(c, cudaMemcpyAsync(out, c->outs.p, 32, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return BP_OK;
}

// ---------------------------------------------------------------------------------------------- range proofs
int bp_rangeproof_verify_reserve(bp_ctx *c, bp_gens *gens, size_t n, size_t m, size_t count, size_t n_batches) {
    if (!c || !gens) return BP_ERR_INVALID_ARGUMENT;
    BUSY_CHECK(c);
    CK(c, cudaSetDevice(c->device));
    size_t k = 0; while (((size_t)1 << k) < n * m) k++;
    rp_geom g{};
    if (rp_param_verdict(gens, 32 * (9 + 2 * k), n, m, &g) != BP_PROOF_OK || !rp_set_group(&g, count, n_batches)) return BP_ERR_INVALID_ARGUMENT;
    CK(c, c->rp_proofs.ensure((size_t)g.count * g.nbatch * g.proof_len)); CK(c, c->rp_commit.ensure((size_t)g.count * g.nbatch * m * 32)); CK(c, c->rp_verdict.ensure((size_t)g.count * g.nbatch * 4));
    int rc = rp_ensure(c, g); if (rc) return rc;
    rc = rp_build_maps(c, gens, g); if (rc) return rc;
    CK(c, cudaStreamSynchronize(c->stream));
    if (c->graph) { cudaGraphExecDestroy(c->graph); c->graph = nullptr; }
    bool prof = c->prof_on; c->prof_on = false;
    uint64_t l0 = c->launches;
    cudaGraph_t graph = nullptr;
    CK(c, cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
    rc = rp_chain(c, gens, g);
    cudaError_t e = cudaStreamEndCapture(c->stream, &graph);
    c->prof_on = prof;
    c->graph_launches = c->launches - l0; c->launches = l0;
    if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
    if (e != cudaSuccess) { c->err = std::string("cudaStreamEndCapture: ") + cudaGetErrorString(e); return BP_ERR_CUDA; }
    e = cudaGraphInstantiate(&c->graph, graph, 0);
    cudaGraphDestroy(graph);
    if (e != cudaSuccess) { c->graph = nullptr; c->err = std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e); return BP_ERR_CUDA; }
    c->graph_key = rp_graph_key(gens, g); c->graph_sig = c->rp.signature();
    // one untimed pass so that the first real call finds module loading, the graph upload and the L2 working set done
    std::vector<uint8_t> zt(BP_TRANSCRIPT_BYTES, 0);
    CK(c, cudaMemsetAsync(c->rp_proofs.p, 0, (size_t)g.count * g.nbatch * g.proof_len, c->stream)); CK(c, cudaMemsetAsync(c->rp_commit.p, 0, (size_t)g.count * g.nbatch * m * 32, c->stream));
    rc = rp_verify_queue(c, gens, g, c->rp_proofs.as<uint8_t>(), c->rp_commit.as<uint8_t>(), zt.data(), nullptr, c->rp_verdict.as<uint32_t>());
    if (rc) return rc;
    CK(c, cudaStreamSynchronize(c->stream));
    return BP_OK;
}

int bp_rangeproof_verify_group_begin(bp_ctx *c, bp_gens *gens, const uint8_t *transcript, const uint8_t *proofs, size_t proof_len, const uint8_t *commitments,
                                     size_t n, size_t m, size_t count, size_t n_batches, const uint8_t *seed) {
    if (!c || !gens || !transcript || !proofs || !commitments || count == 0 || n_batches == 0) return BP_ERR_INVALID_ARGUMENT;
    if (c->vs.active) { c->err = "verify_begin called twice without verify_finish"; return BP_ERR_INVALID_ARGUMENT; }
    if (count * n_batches >= (1u << 24) || n_batches > BP_MAX_GROUP_BATCHES) return BP_ERR_INVALID_ARGUMENT;
    CK(c, cudaSetDevice(c->device));
    rp_geom g{};
    uint8_t pv = rp_param_verdict(gens, proof_len, n, m, &g);
    VerifyState vs; vs.total = (uint32_t)(count * n_batches); vs.n_batches = (uint32_t)n_batches; vs.gens = gens; vs.param_verdict = pv;
    if (pv != BP_PROOF_OK) { vs.active = true; c->vs = vs; return BP_OK; }     // the whole call gets this verdict in _finish
    if (!rp_set_group(&g, count, n_batches)) return BP_ERR_INVALID_ARGUMENT;
    vs.g = g;
    size_t total = vs.total;
    CK(c, c->rp_proofs.ensure(total * proof_len)); CK(c, c->rp_commit.ensure(total * m * 32)); CK(c, c->rp_verdict.ensure(total * 4));
    CK(c, cudaMemcpyAsync(c->rp_proofs.p, proofs, total * proof_len, cudaMemcpyHostToDevice, c->stream));
    CK(c, cudaMemcpyAsync(c->rp_commit.p, commitments, total * m * 32, cudaMemcpyHostToDevice, c->stream));
    int rc = rp_verify_queue(c, gens, g, c->rp_proofs.as<uint8_t>(), c->rp_commit.as<uint8_t>(), transcript, seed, c->rp_verdict.as<uint32_t>());
    if (rc) return rc;
    CK(c, cudaMemcpyAsync(c->h_verdict.p, c->rp_verdict.p, total * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaMemcpyAsync(c->h_flag.p, c->rp.combined.p, (size_t)g.nbatch * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaMemcpyAsync(c->h_flag.as<uint32_t>() + BP_MAX_GROUP_BATCHES, c->rp.batch_ok.p, (size_t)g.nbatch * 4, cudaMemcpyDeviceToHost, c->stream));
    vs.active = true; c->vs = vs;              // only a fully queued verification is pending
    return BP_OK;
}

int bp_rangeproof_verify_group_finish(bp_ctx *c, uint8_t *verdicts, uint8_t *batch_ok) {
    if (!c || !verdicts || !c->vs.active) return BP_ERR_INVALID_ARGUMENT;
    VerifyState vs = c->vs; c->vs.active = false;
    if (vs.param_verdict != BP_PROOF_OK) { memset(verdicts, (int)vs.param_verdict, vs.total); if (batch_ok) memset(batch_ok, 0, vs.n_batches); return BP_OK; }
    CK(c, cudaSetDevice(c->device));
    CK(c, cudaStreamSynchronize(c->stream));
    bool redo = false, contrib_ready = false;
    for (uint32_t b = 0; b < vs.g.nbatch; b++)
        if (c->h_flag.as<uint32_t>()[b] == 0) {            // this batch's combined check failed: find the offenders (chunks of 32, then proof by proof)
            int rc = rp_verify_fallback(c, vs.gens, vs.g, b, c->rp_verdict.as<uint32_t>(), &contrib_ready);
            if (rc) return rc;
            redo = true;
        }
    if (redo) {
        CK(c, cudaMemcpyAsync(c->h_verdict.p, c->rp_verdict.p, (size_t)vs.total * 4, cudaMemcpyDeviceToHost, c->stream));
        CK(c, cudaStreamSynchronize(c->stream));
    }
    for (uint32_t i = 0; i < vs.total; i++) verdicts[i] = (uint8_t)c->h_verdict.as<uint32_t>()[i];
    if (batch_ok) for (uint32_t b = 0; b < vs.g.nbatch; b++) batch_ok[b] = (uint8_t)c->h_flag.as<uint32_t>()[BP_MAX_GROUP_BATCHES + b];
    return BP_OK;
}

int bp_rangeproof_verify_group_device(bp_ctx *c, bp_gens *gens, const uint8_t *transcript, const void *d_proofs, size_t proof_len, const void *d_commitments,
                                      size_t n, size_t m, size_t count, size_t n_batches, const uint8_t *seed, void *d_verdicts_u32, uint32_t *h_batch_ok_pinned) {
    if (!c || !gens || !transcript || !d_proofs || !d_commitments || !d_verdicts_u32) return BP_ERR_INVALID_ARGUMENT;
    BUSY_CHECK(c);
    CK(c, cudaSetDevice(c->device));
    rp_geom g{};
    uint8_t pv = rp_param_verdict(gens, proof_len, n, m, &g);
    if (pv != BP_PROOF_OK || !rp_set_group(&g, count, n_batches)) return BP_ERR_INVALID_ARGUMENT;
    int rc = rp_verify_queue(c, gens, g, (const uint8_t *)d_proofs, (const uint8_t *)d_commitments, transcript, seed, (uint32_t *)d_verdicts_u32);
    if (rc) return rc;
    if (h_batch_ok_pinned) CK(c, cudaMemcpyAsync(h_batch_ok_pinned, c->rp.batch_ok.p, (size_t)g.nbatch * 4, cudaMemcpyDeviceToHost, c->stream));
    return BP_OK;
}

// single-batch forms
int bp_rangeproof_verify_begin(bp_ctx *c, bp_gens *gens, const uint8_t *transcript, const uint8_t *proofs, size_t proof_len, const uint8_t *commitments,
                               size_t n, size_t m, size_t count, const uint8_t *seed) {
    return bp_rangeproof_verify_group_begin(c, gens, transcript, proofs, proof_len, commitments, n, m, count, 1, seed);
}
int bp_rangeproof_verify_finish(bp_ctx *c, uint8_t *verdicts) { return bp_rangeproof_verify_group_finish(c, verdicts, nullptr); }
int bp_rangeproof_verify_batch(bp_ctx *c, bp_gens *gens, const uint8_t *transcript, const uint8_t *proofs, size_t proof_len, const uint8_t *commitments,
                               size_t n, size_t m, size_t count, const uint8_t *seed, uint8_t *verdicts) {
    int rc = bp_rangeproof_verify_begin(c, gens, transcript, proofs, proof_len, commitments, n, m, count, seed);
    if (rc) return rc;
    return bp_rangeproof_verify_finish(c, verdicts);
}
int bp_rangeproof_verify_batch_device(bp_ctx *c, bp_gens *gens, const uint8_t *transcript, const void *d_proofs, size_t proof_len, const void *d_commitments,
                                      size_t n, size_t m, size_t count, const uint8_t *seed, void *d_verdicts_u32, uint32_t *h_batch_ok_pinned) {
    return bp_rangeproof_verify_group_device(c, gens, transcript, d_proofs, proof_len, d_commitments, n, m, count, 1, seed, d_verdicts_u32, h_batch_ok_pinned);
}

// ---------------------------------------------------------------------------------------------- indexed MSMs and the IPP prover session
int bp_msm_indexed_batch(bp_ctx *c, bp_gens *gens, const uint8_t *scalars, const uint32_t *point_idx, const uint8_t *dyn_points, size_t n_dyn,
                         const uint64_t *offsets, size_t n_msm, uint8_t *outs, uint8_t *status) {
    if (!c || !offsets || !outs || n_msm == 0) return BP_ERR_INVALID_ARGUMENT;
    size_t T = offsets[n_msm];
    if (offsets[0] != 0 || T == 0 || T >= (1u << 31) || !scalars || !point_idx) return BP_ERR_INVALID_ARGUMENT;
    BUSY_CHECK(c);
    CK(c, cudaSetDevice(c->device));
    for (size_t t = 0; t < T; t++) {
        uint32_t v = point_idx[t];
        if (v & BP_POINT_DYNAMIC) { if ((v & 0x7fffffffu) >= n_dyn || !dyn_points) return BP_ERR_INVALID_ARGUMENT; }
        else if (!gens || v >= gens->n_points) return BP_ERR_INVALID_ARGUMENT;
    }
    std::vector<uint32_t> off32(n_msm + 1);
    for (size_t j = 0; j <= n_msm; j++) { if (j && offsets[j] < offsets[j - 1]) return BP_ERR_LENGTH_MISMATCH; off32[j] = (uint32_t)offsets[j]; }
    cudaStream_t s = c->stream;
    uint32_t M = (uint32_t)n_msm;
    CK(c, c->in_scalars.ensure(T * 32)); CK(c, c->in_offsets.ensure((n_msm + 1) * 4)); CK(c, c->ix_pidx.ensure(T * 4));
    CK(c, c->outs.ensure(n_msm * 32)); CK(c, c->flags.ensure(n_msm)); CK(c, c->msm_err.ensure((size_t)M * 4)); CK(c, c->results.ensure((size_t)M * sizeof(ge_ext)));
    CK(c, cudaMemcpyAsync(c->in_scalars.p, scalars, T * 32, cudaMemcpyHostToDevice, s));
    CK(c, cudaMemcpyAsync(c->in_offsets.p, off32.data(), (n_msm + 1) * 4, cudaMemcpyHostToDevice, s));
    CK(c, cudaMemcpyAsync(c->ix_pidx.p, point_idx, T * 4, cudaMemcpyHostToDevice, s));
    CK(c, cudaMemsetAsync(c->msm_err.p, 0, (size_t)M * 4, s));
    std::vector<uint8_t> dyn_ok;
    if (n_dyn) {          // per-point flags, not a failure: an invalid point only poisons the MSMs that use it (below)
        CK(c, c->in_points.ensure(n_dyn * 32)); CK(c, c->niels.ensure(n_dyn * sizeof(ge_niels))); CK(c, c->ok.ensure(n_dyn));
        CK(c, cudaMemcpyAsync(c->in_points.p, dyn_points, n_dyn * 32, cudaMemcpyHostToDevice, s));
        LAUNCH(c, KID_DECOMPRESS, k_decompress<<<blocks_for(n_dyn, 128), 128, 0, s>>>(c->in_points.as<uint8_t>(), n_dyn, c->niels.as<ge_niels>(), c->ok.as<uint8_t>()));
        dyn_ok.resize(n_dyn);
        CK(c, cudaMemcpyAsync(dyn_ok.data(), c->ok.p, n_dyn, cudaMemcpyDeviceToHost, s));
    }
    MsmArgs a{c->in_scalars.as<uint8_t>(), c->in_offsets.as<uint32_t>(), M, (uint32_t)T, c->ix_pidx.as<uint32_t>(), gens ? gens->d_table() : nullptr, c->niels.as<ge_niels>(), c->msm_err.as<uint32_t>(), 0};
    int rc = msm_to_bytes(c, a, c->outs.as<uint8_t>(), c->flags.as<uint8_t>());
    if (rc) return rc;
    std::vector<uint8_t> st(n_msm);
    CK(c, cudaMemcpyAsync(outs, c->outs.p, n_msm * 32, cudaMemcpyDeviceToHost, s));
    CK(c, cudaMemcpyAsync(st.data(), c->flags.p, n_msm, cudaMemcpyDeviceToHost, s));
    CK(c, cudaStreamSynchronize(s));
    // an undecodable caller-supplied point poisons the MSMs that use it (optional_multiscalar_mul -> None)
    if (n_dyn)
        for (size_t j = 0; j < n_msm; j++)
            for (size_t t = offsets[j]; t < offsets[j + 1]; t++)
                if ((point_idx[t] & BP_POINT_DYNAMIC) && !dyn_ok[point_idx[t] & 0x7fffffffu] && st[j] == BP_OK) st[j] = BP_ERR_INVALID_POINT;
    if (status) memcpy(status, st.data(), n_msm);
    return BP_OK;
}

// Constant-time form (msm_ct.cuh): table slots only.  Which kernels run, their grids and every copy follow from (T, n_msm, offsets);
// the scalars choose nothing.  Their device copy and the digits recoded from them are cleared on the stream before the call returns.
int bp_msm_indexed_batch_ct(bp_ctx *c, bp_gens *gens, const uint8_t *scalars, const uint32_t *point_idx, const uint64_t *offsets, size_t n_msm,
                            uint8_t *outs, uint8_t *status) {
    if (!c || !offsets || !outs || n_msm == 0) return BP_ERR_INVALID_ARGUMENT;
    size_t T = offsets[n_msm];
    if (offsets[0] != 0 || T == 0 || T >= (1u << 31) || !scalars || !point_idx) return BP_ERR_INVALID_ARGUMENT;
    BUSY_CHECK(c);
    CK(c, cudaSetDevice(c->device));
    if (!gens) return BP_ERR_INVALID_ARGUMENT;
    for (size_t t = 0; t < T; t++) if (point_idx[t] >= gens->n_points) return BP_ERR_INVALID_ARGUMENT;      // dynamic points are not accepted
    std::vector<uint32_t> off32(n_msm + 1);
    for (size_t j = 0; j <= n_msm; j++) { if (j && offsets[j] < offsets[j - 1]) return BP_ERR_LENGTH_MISMATCH; off32[j] = (uint32_t)offsets[j]; }
    // chunks of at most `ch` consecutive terms, never across an MSM boundary; ch grows while the grid would still hold >= 148 x 128 threads,
    // trading parallelism for fewer doublings per term (four per window per chunk)
    uint32_t ch = 1;
    while (ch < 16 && T / (2 * ch) >= 148 * 128) ch *= 2;
    std::vector<uint32_t> bounds;            // [chunk starts (n_chunks) | T | first chunk of each MSM (n_msm + 1)]
    std::vector<uint32_t> msm_first(n_msm + 1);
    for (size_t j = 0; j < n_msm; j++) {
        msm_first[j] = (uint32_t)bounds.size();
        for (uint32_t t = off32[j]; t < off32[j + 1]; t += ch) bounds.push_back(t);
    }
    const uint32_t n_chunks = (uint32_t)bounds.size(); msm_first[n_msm] = n_chunks;
    bounds.push_back((uint32_t)T);
    bounds.insert(bounds.end(), msm_first.begin(), msm_first.end());
    cudaStream_t s = c->stream;
    const uint32_t M = (uint32_t)n_msm;
    CK(c, c->in_scalars.ensure(T * 32)); CK(c, c->in_offsets.ensure((n_msm + 1) * 4)); CK(c, c->ix_pidx.ensure(T * 4));
    CK(c, c->outs.ensure(n_msm * 32)); CK(c, c->flags.ensure(n_msm)); CK(c, c->msm_err.ensure((size_t)M * 4)); CK(c, c->results.ensure((size_t)M * sizeof(ge_ext)));
    CK(c, c->ct_digits.ensure(T * CT_DIGITS)); CK(c, c->ct_tab.ensure(T * CT_TABLE * sizeof(ge_ext)));
    CK(c, c->ct_chunks.ensure(bounds.size() * 4)); CK(c, c->ct_part.ensure((size_t)n_chunks * sizeof(ge_ext)));
    CK(c, cudaMemcpyAsync(c->in_scalars.p, scalars, T * 32, cudaMemcpyHostToDevice, s));
    CK(c, cudaMemcpyAsync(c->in_offsets.p, off32.data(), (n_msm + 1) * 4, cudaMemcpyHostToDevice, s));
    CK(c, cudaMemcpyAsync(c->ix_pidx.p, point_idx, T * 4, cudaMemcpyHostToDevice, s));
    CK(c, cudaMemcpyAsync(c->ct_chunks.p, bounds.data(), bounds.size() * 4, cudaMemcpyHostToDevice, s));
    CK(c, cudaMemsetAsync(c->msm_err.p, 0, (size_t)M * 4, s));
    const uint32_t *d_chunks = c->ct_chunks.as<uint32_t>(), *d_msm_first = d_chunks + n_chunks + 1;
    LAUNCH(c, KID_MSM_CT_RECODE, k_msm_ct_recode<<<blocks_for(T, 128), 128, 0, s>>>(c->in_scalars.as<uint8_t>(), c->in_offsets.as<uint32_t>(), M, (uint32_t)T,
                                                                                    c->ct_digits.as<int8_t>(), c->msm_err.as<uint32_t>()));
    LAUNCH(c, KID_MSM_CT_TABLE, k_msm_ct_table<<<blocks_for(T, 128), 128, 0, s>>>(c->ix_pidx.as<uint32_t>(), (uint32_t)T, gens->d_table(), c->ct_tab.as<ge_ext>()));
    LAUNCH(c, KID_MSM_CT_STRAUS, k_msm_ct_straus<<<blocks_for(n_chunks, 128), 128, 0, s>>>(d_chunks, n_chunks, c->ct_digits.as<int8_t>(), c->ct_tab.as<ge_ext>(), c->ct_part.as<ge_ext>()));
    LAUNCH(c, KID_MSM_CT_REDUCE, k_msm_ct_reduce<<<M, CT_REDUCE_THREADS, 0, s>>>(c->ct_part.as<ge_ext>(), d_msm_first, c->results.as<ge_ext>()));
    LAUNCH(c, KID_COMPRESS, k_compress<<<blocks_for(M, 128), 128, 0, s>>>(c->results.as<ge_ext>(), M, c->outs.as<uint8_t>()));
    LAUNCH(c, KID_SMALL, k_msm_status<<<blocks_for(M, 128), 128, 0, s>>>(c->msm_err.as<uint32_t>(), M, c->flags.as<uint8_t>()));
    // clear_on_drop of the reference's secrets: the scalars and their digits do not outlive the call on the device
    CK(c, cudaMemsetAsync(c->in_scalars.p, 0, T * 32, s));
    CK(c, cudaMemsetAsync(c->ct_digits.p, 0, T * CT_DIGITS, s));
    return msm_copy_out(c, n_msm, outs, status);
}

int bp_ipp_begin_points(bp_ctx *c, const uint8_t *G, const uint8_t *H, size_t N, const uint8_t Q[32], bp_ipp **out) {
    if (!out) return BP_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    if (!c || !G || !H || !Q || N == 0 || (N & (N - 1)) || N >= (1u << 24)) return BP_ERR_INVALID_ARGUMENT;      // power of two (inner_product_proof.rs:67)
    CK(c, cudaSetDevice(c->device));
    std::unique_ptr<bp_ipp> s(new bp_ipp()); s->ctx = c; s->N = (uint32_t)N;
    size_t n_pts = 2 * N + 1;
    CK(c, s->pts.alloc(n_pts * sizeof(ge_niels)));
    cudaStream_t st = c->stream;
    CK(c, c->in_points.ensure(n_pts * 32));
    CK(c, cudaMemcpyAsync(c->in_points.p, G, N * 32, cudaMemcpyHostToDevice, st));
    CK(c, cudaMemcpyAsync(c->in_points.as<uint8_t>() + N * 32, H, N * 32, cudaMemcpyHostToDevice, st));
    CK(c, cudaMemcpyAsync(c->in_points.as<uint8_t>() + 2 * N * 32, Q, 32, cudaMemcpyHostToDevice, st));
    int rc = decompress_checked(c, c->in_points.as<uint8_t>(), n_pts, s->pts.as<ge_niels>());
    if (rc) return rc;
    *out = s.release();
    return BP_OK;
}
void bp_ipp_end(bp_ipp *s) { if (!s) return; cudaSetDevice(s->ctx->device); cudaStreamSynchronize(s->ctx->stream); delete s; }

// one round's two MSMs: L = <sL[0..h), G_R> + <sL[h..2h), H_L> + sL[2h] Q ;  R = <sR[0..h), G_L> + <sR[h..2h), H_R> + sR[2h] Q
// (inner_product_proof.rs:87-113,153-163); h = n_half = current length / 2
int bp_ipp_lr(bp_ipp *s, size_t n_half, const uint8_t *scalars_L, const uint8_t *scalars_R, uint8_t L_out[32], uint8_t R_out[32]) {
    if (!s || !scalars_L || !scalars_R || !L_out || !R_out || n_half == 0 || 2 * n_half > s->N) return BP_ERR_INVALID_ARGUMENT;
    bp_ctx *c = s->ctx; BUSY_CHECK(c); CK(c, cudaSetDevice(c->device));
    size_t h = n_half, per = 2 * h + 1, N = s->N;
    if (check_scalars_canonical(scalars_L, per) || check_scalars_canonical(scalars_R, per)) return BP_ERR_NONCANONICAL_SCALAR;
    std::vector<uint32_t> idx(2 * per), offs = {0, (uint32_t)per, (uint32_t)(2 * per)};
    for (size_t i = 0; i < h; i++) {
        idx[i] = BP_POINT_DYNAMIC | (uint32_t)(h + i);              // G_R
        idx[h + i] = BP_POINT_DYNAMIC | (uint32_t)(N + i);          // H_L
        idx[per + i] = BP_POINT_DYNAMIC | (uint32_t)i;              // G_L
        idx[per + h + i] = BP_POINT_DYNAMIC | (uint32_t)(N + h + i);  // H_R
    }
    idx[2 * h] = idx[per + 2 * h] = BP_POINT_DYNAMIC | (uint32_t)(2 * N);   // Q
    cudaStream_t st = c->stream;
    CK(c, s->scal.ensure(2 * per * 32)); CK(c, s->idx.ensure(std::max<size_t>(2 * per, 2 * N) * 4)); CK(c, s->offs.ensure(16));
    CK(c, c->results.ensure(2 * sizeof(ge_ext))); CK(c, c->outs.ensure(64));
    CK(c, cudaMemcpyAsync(s->scal.p, scalars_L, per * 32, cudaMemcpyHostToDevice, st));
    CK(c, cudaMemcpyAsync(s->scal.as<uint8_t>() + per * 32, scalars_R, per * 32, cudaMemcpyHostToDevice, st));
    CK(c, cudaMemcpyAsync(s->idx.p, idx.data(), 2 * per * 4, cudaMemcpyHostToDevice, st));
    CK(c, cudaMemcpyAsync(s->offs.p, offs.data(), 12, cudaMemcpyHostToDevice, st));
    MsmArgs a{s->scal.as<uint8_t>(), s->offs.as<uint32_t>(), 2, (uint32_t)(2 * per), s->idx.as<uint32_t>(), nullptr, s->pts.as<ge_niels>(), nullptr, 0};
    int rc = msm_to_bytes(c, a, c->outs.as<uint8_t>(), nullptr);
    if (rc) return rc;
    uint8_t lr[64];
    CK(c, cudaMemcpyAsync(lr, c->outs.p, 64, cudaMemcpyDeviceToHost, st)); CK(c, cudaStreamSynchronize(st));
    memcpy(L_out, lr, 32); memcpy(R_out, lr + 32, 32);
    return BP_OK;
}
// G_L[i] = g_lo[i] G_L[i] + g_hi[i] G_R[i] ;  H_L[i] = h_lo[i] H_L[i] + h_hi[i] H_R[i]   (inner_product_proof.rs:124-135,174-179).
// per_index = 1: n_half scalars in each array (first round, factors folded in); 0: one scalar each (u^-1, u / u, u^-1).
int bp_ipp_fold(bp_ipp *s, size_t n_half, const uint8_t *g_lo, const uint8_t *g_hi, const uint8_t *h_lo, const uint8_t *h_hi, int per_index) {
    if (!s || !g_lo || !g_hi || !h_lo || !h_hi || n_half == 0 || 2 * n_half > s->N) return BP_ERR_INVALID_ARGUMENT;
    bp_ctx *c = s->ctx; BUSY_CHECK(c); CK(c, cudaSetDevice(c->device));
    size_t cnt = per_index ? n_half : 1, h = n_half;
    const uint8_t *arrs[4] = {g_lo, g_hi, h_lo, h_hi};
    for (auto a : arrs) if (check_scalars_canonical(a, cnt)) return BP_ERR_NONCANONICAL_SCALAR;
    cudaStream_t st = c->stream;
    CK(c, s->scal.ensure(4 * cnt * 32));
    for (int k = 0; k < 4; k++) CK(c, cudaMemcpyAsync(s->scal.as<uint8_t>() + (size_t)k * cnt * 32, arrs[k], cnt * 32, cudaMemcpyHostToDevice, st));
    uint32_t stride = per_index ? 32 : 0;
    const uint8_t *d = s->scal.as<uint8_t>();
    ge_niels *pts = s->pts.as<ge_niels>();
    LAUNCH(c, KID_IPP_FOLD, k_ipp_fold<<<blocks_for(h, 64), 64, 0, st>>>(pts, (uint32_t)h, d, d + cnt * 32, stride));
    LAUNCH(c, KID_IPP_FOLD, k_ipp_fold<<<blocks_for(h, 64), 64, 0, st>>>(pts + s->N, (uint32_t)h, d + 2 * cnt * 32, d + 3 * cnt * 32, stride));
    CK(c, cudaStreamSynchronize(st));          // the scalar staging buffer is reused by the next round
    return BP_OK;
}

// ---------------------------------------------------------------------------------------------- inner-product prover, device-resident state
int bp_ippx_begin(bp_ctx *c, bp_gens *gens, size_t n, size_t m, size_t n_proofs, const uint8_t *Q, const uint8_t *Gf, const uint8_t *Hf, const uint8_t *a, const uint8_t *b, bp_ippx **out) {
    if (!out) return BP_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    if (!gens || !Q || !a || !b || n == 0 || m == 0 || n > gens->cap || m > gens->parties) return BP_ERR_INVALID_ARGUMENT;
    size_t N = n * m;
    std::unique_ptr<bp_ippx> s;
    int rc = ippx_alloc(c, N, n_proofs, s); if (rc) return rc;
    s->d_static = gens->d_table();
    std::vector<uint32_t> idx(2 * N);
    for (size_t q = 0; q < N; q++) {          // BulletproofGens::G(n, m) / H(n, m) iterator order
        idx[q] = (uint32_t)gens_slot<size_t>(0, q / n, q % n, gens->cap, gens->parties);
        idx[N + q] = (uint32_t)gens_slot<size_t>(1, q / n, q % n, gens->cap, gens->parties);
    }
    CK(c, cudaMemcpyAsync(s->gidx.p, idx.data(), N * 4, cudaMemcpyHostToDevice, c->stream)); CK(c, cudaMemcpyAsync(s->hidx.p, idx.data() + N, N * 4, cudaMemcpyHostToDevice, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    rc = ippx_load(s.get(), Q, Gf, Hf, a, b);
    if (rc) return rc;
    *out = s.release();
    return BP_OK;
}
int bp_ippx_begin_points(bp_ctx *c, const uint8_t *G, const uint8_t *H, size_t N, size_t n_proofs, const uint8_t *Q, const uint8_t *Gf, const uint8_t *Hf, const uint8_t *a, const uint8_t *b, bp_ippx **out) {
    if (!out) return BP_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    if (!G || !H || !Q || !a || !b) return BP_ERR_INVALID_ARGUMENT;
    std::unique_ptr<bp_ippx> s;
    int rc = ippx_alloc(c, N, n_proofs, s); if (rc) return rc;
    cudaStream_t st = c->stream;
    CK(c, s->own_pts.alloc(2 * N * sizeof(ge_niels)));
    s->d_static = s->own_pts.as<ge_niels>();
    std::vector<uint32_t> idx(2 * N);
    for (size_t q = 0; q < 2 * N; q++) idx[q] = (uint32_t)q;
    CK(c, c->in_points.ensure(2 * N * 32));
    CK(c, cudaMemcpyAsync(c->in_points.p, G, N * 32, cudaMemcpyHostToDevice, st)); CK(c, cudaMemcpyAsync(c->in_points.as<uint8_t>() + N * 32, H, N * 32, cudaMemcpyHostToDevice, st));
    CK(c, cudaMemcpyAsync(s->gidx.p, idx.data(), N * 4, cudaMemcpyHostToDevice, st)); CK(c, cudaMemcpyAsync(s->hidx.p, idx.data() + N, N * 4, cudaMemcpyHostToDevice, st));
    rc = decompress_checked(c, c->in_points.as<uint8_t>(), 2 * N, s->own_pts.as<ge_niels>());
    if (rc) return rc;
    rc = ippx_load(s.get(), Q, Gf, Hf, a, b);
    if (rc) return rc;
    *out = s.release();
    return BP_OK;
}
void bp_ippx_end(bp_ippx *s) { if (!s) return; cudaSetDevice(s->ctx->device); cudaStreamSynchronize(s->ctx->stream); delete s; }
size_t bp_ippx_current_len(const bp_ippx *s) { return s ? s->n : 0; }
// L and R of the current round for every proof (inner_product_proof.rs:87-113 / 153-163): LR_out = n_proofs x (L | R) compressed; synchronises
int bp_ippx_round(bp_ippx *s, uint8_t *LR_out) {
    if (!s || !LR_out || s->n < 2) return BP_ERR_INVALID_ARGUMENT;
    bp_ctx *c = s->ctx; BUSY_CHECK(c); CK(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream; ippx_geom g{s->N, s->B, s->n};
    uint32_t M = 2 * s->B, T = M * (s->N + 1);
    LAUNCH(c, KID_SMALL, k_ippx_inner<<<M, 128, 0, st>>>(g, s->a.as<sc>(), s->b.as<sc>(), s->scal.as<uint8_t>()));
    LAUNCH(c, KID_SMALL, k_ippx_rows<<<blocks_for((size_t)s->B * s->N, 128), 128, 0, st>>>(g, s->a.as<sc>(), s->b.as<sc>(), s->cG.as<sc>(), s->cH.as<sc>(), s->gidx.as<uint32_t>(), s->hidx.as<uint32_t>(),
                                                                                          s->scal.as<uint8_t>(), s->pidx.as<uint32_t>()));
    CK(c, c->results.ensure((size_t)M * sizeof(ge_ext)));
    MsmArgs a{s->scal.as<uint8_t>(), s->offs.as<uint32_t>(), M, T, s->pidx.as<uint32_t>(), s->d_static, s->d_q.as<ge_niels>(), nullptr, 0};
    int rc = msm_to_bytes(c, a, s->outs.as<uint8_t>(), nullptr);
    if (rc) return rc;
    CK(c, cudaMemcpyAsync(LR_out, s->outs.p, (size_t)M * 32, cudaMemcpyDeviceToHost, st)); CK(c, cudaStreamSynchronize(st));
    return BP_OK;
}
// apply the challenges u (and their inverses), one pair per proof; halves the current length
int bp_ippx_fold(bp_ippx *s, const uint8_t *u, const uint8_t *u_inv) {
    if (!s || !u || !u_inv || s->n < 2) return BP_ERR_INVALID_ARGUMENT;
    bp_ctx *c = s->ctx; BUSY_CHECK(c); CK(c, cudaSetDevice(c->device));
    if (check_scalars_canonical(u, s->B) || check_scalars_canonical(u_inv, s->B)) return BP_ERR_NONCANONICAL_SCALAR;
    cudaStream_t st = c->stream; ippx_geom g{s->N, s->B, s->n};
    uint8_t *din = s->in.as<uint8_t>();
    CK(c, cudaMemcpyAsync(din, u, (size_t)s->B * 32, cudaMemcpyHostToDevice, st)); CK(c, cudaMemcpyAsync(din + (size_t)s->B * 32, u_inv, (size_t)s->B * 32, cudaMemcpyHostToDevice, st));
    LAUNCH(c, KID_IPP_FOLD, k_ippx_fold<<<blocks_for((size_t)s->B * s->N, 128), 128, 0, st>>>(g, din, din + (size_t)s->B * 32, s->a.as<sc>(), s->b.as<sc>(), s->cG.as<sc>(), s->cH.as<sc>()));
    CK(c, cudaStreamSynchronize(st));          // the staging buffer is reused by the next call
    s->n >>= 1;
    return BP_OK;
}
// the final a, b (inner_product_proof.rs:187-192): ab_out = n_proofs x (a | b)
int bp_ippx_finish(bp_ippx *s, uint8_t *ab_out) {
    if (!s || !ab_out || s->n != 1) return BP_ERR_INVALID_ARGUMENT;
    bp_ctx *c = s->ctx; BUSY_CHECK(c); CK(c, cudaSetDevice(c->device));
    ippx_geom g{s->N, s->B, s->n};
    LAUNCH(c, KID_SMALL, k_ippx_final<<<blocks_for(s->B, 128), 128, 0, c->stream>>>(g, s->a.as<sc>(), s->b.as<sc>(), s->outs.as<uint8_t>()));
    CK(c, cudaMemcpyAsync(ab_out, s->outs.p, (size_t)s->B * 64, cudaMemcpyDeviceToHost, c->stream)); CK(c, cudaStreamSynchronize(c->stream));
    return BP_OK;
}

// ---------------------------------------------------------------------------------------------- per-kernel timing
int bp_prof_enable(bp_ctx *c, int on) {
    if (!c) return BP_ERR_INVALID_ARGUMENT;
    for (ProfRec &r : c->prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    c->prof.clear(); c->prof_on = on != 0; return BP_OK;
}
int bp_prof_kernel_count(void) { return KID_COUNT; }
const char *bp_prof_kernel_name(int kid) { return kid >= 0 && kid < KID_COUNT ? KERNEL_NAMES[kid] : ""; }
// synchronises the stream, adds up the CUDA-event durations recorded since the last report; ms/counts have bp_prof_kernel_count() entries
int bp_prof_report(bp_ctx *c, double *ms, uint64_t *counts) {
    if (!c || !ms || !counts) return BP_ERR_INVALID_ARGUMENT;
    CK(c, cudaSetDevice(c->device)); CK(c, cudaStreamSynchronize(c->stream));
    for (int i = 0; i < KID_COUNT; i++) { ms[i] = 0; counts[i] = 0; }
    for (ProfRec &r : c->prof) { float t = 0; if (cudaEventElapsedTime(&t, r.a, r.b) == cudaSuccess) { ms[r.kid] += t; counts[r.kid]++; } cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    c->prof.clear();
    return BP_OK;
}
// per-launch records since the last report/enable: start and end in ms relative to the first record of `ref` (a context of the
// same device whose profiling was enabled first); synchronises both streams.  Diagnostic for multi-stream overlap.
int bp_prof_timeline(bp_ctx *c, bp_ctx *ref, int *kernel_ids, double *start_ms, double *end_ms, size_t cap, size_t *n_out) {
    if (!c || !ref || !kernel_ids || !start_ms || !end_ms || !n_out) return BP_ERR_INVALID_ARGUMENT;
    CK(c, cudaSetDevice(c->device)); CK(c, cudaStreamSynchronize(c->stream)); CK(c, cudaStreamSynchronize(ref->stream));
    if (ref->prof.empty()) return BP_ERR_INVALID_ARGUMENT;
    size_t n = 0;
    for (ProfRec &r : c->prof) {
        if (n >= cap) break;
        float a = 0, b = 0;
        if (cudaEventElapsedTime(&a, ref->prof[0].a, r.a) != cudaSuccess || cudaEventElapsedTime(&b, ref->prof[0].a, r.b) != cudaSuccess) continue;
        kernel_ids[n] = r.kid; start_ms[n] = a; end_ms[n] = b; n++;
    }
    *n_out = n;
    return BP_OK;
}
// copy the resident generator table to / from another device buffer (e.g. a torch tensor used for the NCCL broadcast)
int bp_gens_table_export(bp_gens *g, void *d_dst) {
    if (!g || !d_dst) return BP_ERR_INVALID_ARGUMENT;
    bp_ctx *c = g->ctx; CK(c, cudaSetDevice(c->device));
    CK(c, cudaMemcpyAsync(d_dst, g->d_table(), g->n_points * sizeof(ge_niels), cudaMemcpyDeviceToDevice, c->stream)); CK(c, cudaStreamSynchronize(c->stream)); return BP_OK;
}
int bp_gens_table_import(bp_gens *g, const void *d_src) {
    if (!g || !d_src) return BP_ERR_INVALID_ARGUMENT;
    bp_ctx *c = g->ctx; CK(c, cudaSetDevice(c->device));
    CK(c, cudaMemcpyAsync(g->d_table(), d_src, g->n_points * sizeof(ge_niels), cudaMemcpyDeviceToDevice, c->stream)); CK(c, cudaStreamSynchronize(c->stream)); return BP_OK;
}

// ---------------------------------------------------------------------------------------------- host helpers
// merlin::Transcript for hosts that do not have the Rust crate (the Python harness, C++ callers):
// same STROBE code the device kernels use, compiled for the host.  Pure byte shuffling, no curve math.
void bp_transcript_new(const uint8_t *label, size_t len, uint8_t out[BP_TRANSCRIPT_BYTES]) { alignas(8) uint8_t st[200]; merlin_t m; m.st = st; merlin_init(m, label, (uint32_t)len); merlin_store(out, m); }
void bp_transcript_append_message(uint8_t state[BP_TRANSCRIPT_BYTES], const char *label, const uint8_t *msg, size_t len) {
    alignas(8) uint8_t st[200]; merlin_t m; m.st = st; merlin_load(m, state); merlin_append(m, label, msg, (uint32_t)len); merlin_store(state, m);
}
void bp_transcript_append_u64(uint8_t state[BP_TRANSCRIPT_BYTES], const char *label, uint64_t x) { alignas(8) uint8_t st[200]; merlin_t m; m.st = st; merlin_load(m, state); merlin_append_u64(m, label, x); merlin_store(state, m); }
void bp_transcript_challenge_bytes(uint8_t state[BP_TRANSCRIPT_BYTES], const char *label, uint8_t *out, size_t len) {
    alignas(8) uint8_t st[200]; merlin_t m; m.st = st; merlin_load(m, state); merlin_challenge(m, label, out, (uint32_t)len); merlin_store(state, m);
}

// test hook: element-wise field operation on the device (pins the PTX carry chains of fe.cuh)
__global__ void k_debug_fe(int op, const uint8_t *a, const uint8_t *b, size_t n, uint8_t *out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t ab[32], bb[32]; ld32(ab, a + 32 * i); ld32(bb, b + 32 * i);
    fe x = fe_frombytes_raw(ab), y = fe_frombytes_raw(bb), r;
    switch (op) {
        case 0: r = fe_add(x, y); break;
        case 1: r = fe_sub(x, y); break;
        case 2: r = fe_mul(x, y); break;
        case 3: r = fe_invert(x); break;
        case 4: r = fe_pow22523(x); break;
        case 5: r = fe_neg(x); break;
        case 7: r = fe_mul(fe_add(x, y), fe_sub(x, y)); break;      // chained, unreduced intermediates
        default: r = fe_sq(x);
    }
    uint8_t o[32]; fe_tobytes(o, r); st32(out + 32 * i, o);
}
int bp_debug_fe_op(bp_ctx *c, int op, const uint8_t *a, const uint8_t *b, size_t n, uint8_t *out) {
    if (!c || !a || !b || !out || n == 0) return BP_ERR_INVALID_ARGUMENT;
    CK(c, cudaSetDevice(c->device));
    CK(c, c->in_scalars.ensure(n * 32)); CK(c, c->in_points.ensure(n * 32)); CK(c, c->outs.ensure(n * 32));
    CK(c, cudaMemcpyAsync(c->in_scalars.p, a, n * 32, cudaMemcpyHostToDevice, c->stream));
    CK(c, cudaMemcpyAsync(c->in_points.p, b, n * 32, cudaMemcpyHostToDevice, c->stream));
    LAUNCH(c, KID_SMALL, k_debug_fe<<<blocks_for(n, 128), 128, 0, c->stream>>>(op, c->in_scalars.as<uint8_t>(), c->in_points.as<uint8_t>(), n, c->outs.as<uint8_t>()));
    CK(c, cudaMemcpyAsync(out, c->outs.p, n * 32, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return BP_OK;
}

}  // extern "C"
