// Device kernels of the MSM engine (sm_100a).  One thread = one independent point / bucket /
// scalar operation; a warp therefore carries 32 independent chains of the 8x32-bit-limb field
// arithmetic in fe.cuh.  The work is integer-pipe bound (IMAD.WIDE), not HBM bound: one 64-byte
// MSM term buys ~W mixed additions = W*7 field multiplications = W*7*72 wide multiplies.
#pragma once
#include <cuda_runtime.h>
#include "ge.cuh"
#include "sc.cuh"
#include "merlin.cuh"
#include "rp.cuh"
#include "msm_common.cuh"
#include "msm_ct.cuh"

#define BP_POINT_DYNAMIC 0x80000000u     // point_idx flag: index into the per-call (dynamic) point array

// Slot of G[party][index] (which = 0) or H[party][index] (which = 1) in the generator table [B_blinding, B, G[party][i].., H[party][i]..].
// BulletproofGens::G(n, m) / H(n, m) visit term q at party q / n, index q % n (generators.rs:207-259).
template <class U> __host__ __device__ inline U gens_slot(U which, U party, U index, U cap, U parties) { return 2 + (which * parties + party) * cap + index; }

// ------------------------------------------------------------------ vector load/store helpers
__device__ __forceinline__ void ld32(uint8_t dst[32], const uint8_t *src) {       // 32 B, 16-B aligned
    const uint4 *p = reinterpret_cast<const uint4 *>(src);
    uint4 a = __ldg(p), b = __ldg(p + 1);
    uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    memcpy(dst, w, 32);
}
__device__ __forceinline__ void ld32_any(uint8_t dst[32], const uint8_t *src) {   // any alignment (proof bytes)
    if ((reinterpret_cast<uintptr_t>(src) & 15) == 0) { ld32(dst, src); return; }
    if ((reinterpret_cast<uintptr_t>(src) & 3) == 0) { const uint32_t *p = reinterpret_cast<const uint32_t *>(src); uint32_t w[8]; for (int i = 0; i < 8; i++) w[i] = __ldg(p + i); memcpy(dst, w, 32); return; }
    for (int i = 0; i < 32; i++) dst[i] = src[i];
}
__device__ __forceinline__ void st32(uint8_t *dst, const uint8_t src[32]) {
    uint32_t w[8]; memcpy(w, src, 32);
    uint4 *p = reinterpret_cast<uint4 *>(dst);
    p[0] = make_uint4(w[0], w[1], w[2], w[3]); p[1] = make_uint4(w[4], w[5], w[6], w[7]);
}
__device__ __forceinline__ fe ld_fe(const fe *p) {
    const uint4 *q = reinterpret_cast<const uint4 *>(p); uint4 a = q[0], b = q[1];
    fe r; r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w; r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w; return r;
}
__device__ __forceinline__ fe ldg_fe(const fe *p) {
    const uint4 *q = reinterpret_cast<const uint4 *>(p); uint4 a = __ldg(q), b = __ldg(q + 1);
    fe r; r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w; r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w; return r;
}
__device__ __forceinline__ void st_fe(fe *p, const fe &v) {
    uint4 *q = reinterpret_cast<uint4 *>(p);
    q[0] = make_uint4(v.v[0], v.v[1], v.v[2], v.v[3]); q[1] = make_uint4(v.v[4], v.v[5], v.v[6], v.v[7]);
}
__device__ __forceinline__ ge_niels ldg_niels(const ge_niels *p) { ge_niels r; r.ypx = ldg_fe(&p->ypx); r.ymx = ldg_fe(&p->ymx); r.xy2d = ldg_fe(&p->xy2d); return r; }
__device__ __forceinline__ void st_niels(ge_niels *p, const ge_niels &v) { st_fe(&p->ypx, v.ypx); st_fe(&p->ymx, v.ymx); st_fe(&p->xy2d, v.xy2d); }
__device__ __forceinline__ ge_ext ld_ext(const ge_ext *p) { ge_ext r; r.X = ld_fe(&p->X); r.Y = ld_fe(&p->Y); r.Z = ld_fe(&p->Z); r.T = ld_fe(&p->T); return r; }
__device__ __forceinline__ void st_ext(ge_ext *p, const ge_ext &v) { st_fe(&p->X, v.X); st_fe(&p->Y, v.Y); st_fe(&p->Z, v.Z); st_fe(&p->T, v.T); }

__device__ __forceinline__ ge_ext shfl_down_ext(const ge_ext &p, int d) {
    ge_ext r;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        r.X.v[i] = __shfl_down_sync(0xffffffffu, p.X.v[i], d); r.Y.v[i] = __shfl_down_sync(0xffffffffu, p.Y.v[i], d);
        r.Z.v[i] = __shfl_down_sync(0xffffffffu, p.Z.v[i], d); r.T.v[i] = __shfl_down_sync(0xffffffffu, p.T.v[i], d);
    }
    return r;
}

// ------------------------------------------------------------------ TMA staging of the streaming byte arrays
// The scalar and compressed-point arrays are read once, front to back.  Each block stages its contiguous tile
// (32 B per thread) into shared memory with ONE bulk asynchronous copy (cp.async.bulk: the TMA engine, SASS UBLKCP)
// signalled through an mbarrier, instead of one 2x128-bit global load pair per thread; threads then read their
// record from shared memory.  src must be 16-byte aligned, bytes a multiple of 16 (records are 32 B).
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void tma_stage_tile(void *smem_dst, const void *gsrc, uint32_t bytes, uint64_t *bar) {
    uint32_t b = smem_u32(bar);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(b));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(b), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(b) : "memory");
    }
    uint32_t done;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(done) : "r"(b) : "memory");
    } while (!done);
}
// Two-source form for the per-proof kernels: a block's slice of the proof array and of the commitment array (both contiguous,
// 16-byte aligned when the caller's buffers are) land in shared memory through two bulk copies signalled on one mbarrier; the
// threads then take their 32-byte fields -- at offsets that are not 16-byte aligned in general -- from shared memory.
// Falls back to a cooperative copy for buffers that are not 16-byte aligned.
__device__ __forceinline__ void tma_stage_two(uint8_t *dst_a, const uint8_t *src_a, uint32_t bytes_a, uint8_t *dst_b, const uint8_t *src_b, uint32_t bytes_b, uint64_t *bar) {
    const bool aligned = ((reinterpret_cast<uintptr_t>(src_a) | reinterpret_cast<uintptr_t>(src_b) | bytes_a | bytes_b) & 15) == 0;
    if (!aligned) {
        for (uint32_t i = threadIdx.x; i < bytes_a; i += blockDim.x) dst_a[i] = src_a[i];
        for (uint32_t i = threadIdx.x; i < bytes_b; i += blockDim.x) dst_b[i] = src_b[i];
        __syncthreads();
        return;
    }
    uint32_t b = smem_u32(bar);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(b));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(b), "r"(bytes_a + bytes_b) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(smem_u32(dst_a)), "l"(src_a), "r"(bytes_a), "r"(b) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(smem_u32(dst_b)), "l"(src_b), "r"(bytes_b), "r"(b) : "memory");
    }
    uint32_t done;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(done) : "r"(b) : "memory");
    } while (!done);
}
__device__ __forceinline__ void lds32(uint8_t dst[32], const uint8_t *smem_src) {
    const uint4 *p = reinterpret_cast<const uint4 *>(smem_src);
    uint4 a = p[0], b = p[1];
    uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    memcpy(dst, w, 32);
}

// ------------------------------------------------------------------ K1: batched Ristretto decompress
// in: n x 32 B compressed.  out: n affine-Niels points (identity when invalid), ok[i] in {0,1}.
__global__ void __launch_bounds__(128) k_decompress(const uint8_t *__restrict__ in, size_t n, ge_niels *__restrict__ out, uint8_t *__restrict__ ok) {
    __shared__ __align__(128) uint8_t tile[128 * 32];
    __shared__ __align__(8) uint64_t bar;
    size_t base = (size_t)blockIdx.x * blockDim.x, i = base + threadIdx.x;
    uint32_t cnt = (uint32_t)min((size_t)blockDim.x, n - base);
    tma_stage_tile(tile, in + 32 * base, 32u * cnt, &bar);
    if (i >= n) return;
    uint8_t s[32]; lds32(s, tile + 32 * threadIdx.x);
    fe x, y; bool valid = ge_decode(x, y, s);
    ge_niels q = valid ? ge_to_niels_affine(x, y) : ge_niels_identity();
    st_niels(out + i, q);
    if (ok) ok[i] = valid ? 1 : 0;
}

// ------------------------------------------------------------------ K3: batched compress / identity test
__global__ void __launch_bounds__(128) k_compress(const ge_ext *__restrict__ in, size_t n, uint8_t *__restrict__ out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t s[32]; ge_encode(s, ld_ext(in + i)); st32(out + 32 * i, s);
}

// ------------------------------------------------------------------ K7: from_uniform_bytes (generator chain)
// in: n x 64 B.  out: affine-Niels table entry and/or compressed bytes.
__global__ void __launch_bounds__(128) k_from_uniform(const uint8_t *__restrict__ in, size_t n, ge_niels *__restrict__ out_niels, uint8_t *__restrict__ out_comp) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t u[64]; ld32(u, in + 64 * i); ld32(u + 32, in + 64 * i + 32);
    ge_ext p = ge_from_uniform(u);
    if (out_comp) { uint8_t s[32]; ge_encode(s, p); st32(out_comp + 32 * i, s); }
    if (out_niels) { fe zi = fe_invert(p.Z); st_niels(out_niels + i, ge_to_niels_affine(fe_mul(p.X, zi), fe_mul(p.Y, zi))); }
}
__global__ void __launch_bounds__(128) k_niels_to_compressed(const ge_niels *__restrict__ in, size_t n, uint8_t *__restrict__ out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t s[32]; ge_encode(s, ge_from_niels(ldg_niels(in + i))); st32(out + 32 * i, s);
}

// ------------------------------------------------------------------ K2: Pippenger bucket pipeline
// A batch of n_msm MSMs over a flat term array.  "segment" = (msm, window); every segment owns nb =
// 2^(c-1) buckets and a slice of `sorted` with room for all terms of its MSM:
//     seg = msm*W + w,   slice base = W*offsets[msm] + w*len,  len = offsets[msm+1]-offsets[msm].
// Buckets are accumulated by one thread each, except "heavy" ones (size >= heavy_min, chosen by the host as a multiple
// of the mean bucket size): k_msm_order lists those and k_msm_accumulate_heavy gives each a whole block.  Heavy buckets
// are not an adversarial corner only: scalars are < l ~ 2^252, so when c*(W-1) = 252 (c = 9, 12, ...) the top window
// holds nothing but the recoding carry and HALF of all terms land in its bucket 0.
__device__ __forceinline__ size_t msm_slice_base(uint32_t o0, uint32_t len, uint32_t w, int W) {
    return (size_t)W * (size_t)o0 + (size_t)w * (size_t)len;
}
__device__ __forceinline__ uint32_t msm_of_term(const uint32_t *__restrict__ offsets, uint32_t n_msm, uint32_t t) {
    uint32_t lo = 0, hi = n_msm;            // largest j with offsets[j] <= t
    while (hi - lo > 1) { uint32_t mid = (lo + hi) >> 1; if (__ldg(offsets + mid) <= t) lo = mid; else hi = mid; }
    return lo;
}

// pass 1: histogram.  One thread per term; scalars are 32-byte canonical little-endian.
__global__ void __launch_bounds__(256) k_msm_count(const uint8_t *__restrict__ scalars, const uint32_t *__restrict__ offsets, uint32_t n_msm, uint32_t T,
                                                   int c, int W, uint32_t *__restrict__ counts, uint32_t *__restrict__ msm_err) {
    __shared__ __align__(128) uint8_t tile[256 * 32];
    __shared__ __align__(8) uint64_t bar;
    uint32_t base = blockIdx.x * blockDim.x, t = base + threadIdx.x;
    tma_stage_tile(tile, scalars + 32 * (size_t)base, 32u * min(blockDim.x, T - base), &bar);
    if (t >= T) return;
    uint8_t sb[32]; lds32(sb, tile + 32 * threadIdx.x);
    sc s = sc_load(sb);
    uint32_t msm = n_msm == 1 ? 0u : msm_of_term(offsets, n_msm, t);
    if (sc_geq_l(s)) { if (msm_err) atomicOr(msm_err + msm, 2u); return; }       // non-canonical scalar
    msm_wide r = msm_recode(s.v, c, W);
    uint32_t nb = 1u << (c - 1);
    for (int w = 0; w < W; w++) {
        int d = msm_digit(r, w, c);
        if (d == 0) continue;
        uint32_t b = (uint32_t)(d < 0 ? -d : d) - 1u;
        atomicAdd(counts + ((size_t)msm * W + w) * nb + b, 1u);
    }
}
// pass 2: per-segment exclusive scan of the bucket counts (block per segment); cursor starts as a copy
#define MSM_SIZE_BINS 256        // bucket sizes are clamped to MSM_SIZE_BINS-1 for the load-balancing order
__global__ void __launch_bounds__(256) k_msm_scan(const uint32_t *__restrict__ counts, uint32_t nb, uint32_t *__restrict__ starts, uint32_t *__restrict__ cursor,
                                                  uint32_t *__restrict__ size_hist) {
    __shared__ uint32_t warp_sums[8];
    __shared__ uint32_t hist[MSM_SIZE_BINS];
    for (uint32_t i = threadIdx.x; i < MSM_SIZE_BINS; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    size_t seg = blockIdx.x;
    const uint32_t *cnt = counts + seg * nb; uint32_t *st = starts + seg * nb, *cu = cursor + seg * nb;
    uint32_t per = (nb + blockDim.x - 1) / blockDim.x;
    uint32_t lo = threadIdx.x * per, hi = min(lo + per, nb);
    uint32_t local = 0;
    for (uint32_t i = lo; i < hi; i++) local += cnt[i];
    // block exclusive scan of `local`
    uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5, v = local;
    for (int d = 1; d < 32; d <<= 1) { uint32_t o = __shfl_up_sync(0xffffffffu, v, d); if (lane >= (uint32_t)d) v += o; }
    if (lane == 31) warp_sums[wid] = v;
    __syncthreads();
    uint32_t base = 0;
    for (uint32_t k = 0; k < wid; k++) base += warp_sums[k];
    uint32_t run = base + v - local;
    for (uint32_t i = lo; i < hi; i++) { uint32_t c_ = cnt[i]; st[i] = run; cu[i] = run; run += c_; atomicAdd(&hist[MSM_SIZE_BINS - 1 - min(c_, (uint32_t)MSM_SIZE_BINS - 1)], 1u); }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < MSM_SIZE_BINS; i += blockDim.x) if (hist[i]) atomicAdd(size_hist + i, hist[i]);
}
// load-balancing order: bucket ids sorted by decreasing size (counting sort over the size histogram), so that the 32
// buckets a warp accumulates have (nearly) equal lengths and the longest buckets start first
__global__ void __launch_bounds__(256) k_msm_order(const uint32_t *__restrict__ counts, size_t n_buckets, const uint32_t *__restrict__ size_hist,
                                                   uint32_t *__restrict__ bin_cursor, uint32_t *__restrict__ order, uint32_t heavy_min,
                                                   uint32_t *__restrict__ heavy_n, uint32_t *__restrict__ heavy) {
    __shared__ uint32_t base[MSM_SIZE_BINS];
    __shared__ uint32_t wsum[8];
    __shared__ uint32_t local[MSM_SIZE_BINS];          // this block's buckets per bin, then the block's base within the bin
    {   // exclusive scan of the 256-bin histogram, redundantly per block
        uint32_t v = size_hist[threadIdx.x], lane = threadIdx.x & 31, wid = threadIdx.x >> 5, x = v;
        for (int d = 1; d < 32; d <<= 1) { uint32_t o = __shfl_up_sync(0xffffffffu, x, d); if (lane >= (uint32_t)d) x += o; }
        if (lane == 31) wsum[wid] = x;
        local[threadIdx.x] = 0;
        __syncthreads();
        uint32_t b = 0; for (uint32_t k = 0; k < wid; k++) b += wsum[k];
        base[threadIdx.x] = b + x - v;
        __syncthreads();
    }
    // rank within (block, bin) through shared-memory atomics, then ONE global atomic per non-empty bin of the block: the buckets of a
    // window have nearly equal sizes, so per-bucket global atomics on a handful of bin cursors serialise (46 us for 786k buckets)
    size_t gb = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool live = gb < n_buckets;
    uint32_t cnt = live ? counts[gb] : 0;
    uint32_t bin = MSM_SIZE_BINS - 1 - min(cnt, (uint32_t)MSM_SIZE_BINS - 1);
    uint32_t rank = live ? atomicAdd(&local[bin], 1u) : 0;
    __syncthreads();
    { uint32_t mine = local[threadIdx.x]; __syncthreads(); local[threadIdx.x] = mine ? atomicAdd(bin_cursor + threadIdx.x, mine) : 0; }
    __syncthreads();
    if (!live) return;
    order[base[bin] + local[bin] + rank] = (uint32_t)gb;
    if (cnt >= heavy_min) heavy[atomicAdd(heavy_n, 1u)] = (uint32_t)gb;
}
// pass 3: scatter term ids (sign in bit 31) into their bucket's slice
__global__ void __launch_bounds__(256) k_msm_scatter(const uint8_t *__restrict__ scalars, const uint32_t *__restrict__ offsets, uint32_t n_msm, uint32_t T,
                                                     int c, int W, uint32_t *__restrict__ cursor, uint32_t *__restrict__ sorted) {
    __shared__ __align__(128) uint8_t tile[256 * 32];
    __shared__ __align__(8) uint64_t bar;
    uint32_t base = blockIdx.x * blockDim.x, t = base + threadIdx.x;
    tma_stage_tile(tile, scalars + 32 * (size_t)base, 32u * min(blockDim.x, T - base), &bar);
    if (t >= T) return;
    uint8_t sb[32]; lds32(sb, tile + 32 * threadIdx.x);
    sc s = sc_load(sb);
    if (sc_geq_l(s)) return;
    uint32_t msm = n_msm == 1 ? 0u : msm_of_term(offsets, n_msm, t);
    uint32_t o0 = __ldg(offsets + msm), len = __ldg(offsets + msm + 1) - o0;
    msm_wide r = msm_recode(s.v, c, W);
    uint32_t nb = 1u << (c - 1);
    for (int w = 0; w < W; w++) {
        int d = msm_digit(r, w, c);
        if (d == 0) continue;
        uint32_t b = (uint32_t)(d < 0 ? -d : d) - 1u;
        uint32_t pos = atomicAdd(cursor + ((size_t)msm * W + w) * nb + b, 1u);
        sorted[msm_slice_base(o0, len, (uint32_t)w, W) + pos] = t | (d < 0 ? 0x80000000u : 0u);
    }
}
// heavy buckets (size >= heavy_min, listed by k_msm_order): one 128-thread block per bucket, grid-stride over the list: threads take
// strided entries, then a shuffle tree + one shared-memory round add the partial sums.  Runs in the first blocks of k_msm_accumulate's
// grid (a separate launch would wait for an SM with a free block slot behind the wide kernels of the other groups in flight).
#define MSM_ACC_THREADS 128
__device__ __noinline__ void msm_heavy_role(const uint32_t *__restrict__ starts, const uint32_t *__restrict__ ends, const uint32_t *__restrict__ sorted,
                                            const uint32_t *__restrict__ offsets, const uint32_t *__restrict__ heavy_n, const uint32_t *__restrict__ heavy, int W, uint32_t nb,
                                            const uint32_t *__restrict__ point_idx, const ge_niels *__restrict__ pts_static, const ge_niels *__restrict__ pts_dynamic,
                                            ge_ext *__restrict__ buckets, uint32_t first, uint32_t stride) {
    __shared__ ge_ext sm[MSM_ACC_THREADS / 32];
    uint32_t n_heavy = *heavy_n, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (uint32_t h = first; h < n_heavy; h += stride) {
        size_t gb = heavy[h];
        size_t seg = gb / nb; uint32_t msm = (uint32_t)(seg / W), w = (uint32_t)(seg % W);
        uint32_t o0 = __ldg(offsets + msm), len = __ldg(offsets + msm + 1) - o0;
        const uint32_t *slice = sorted + msm_slice_base(o0, len, w, W);
        uint32_t lo = starts[gb], hi = ends[gb];
        ge_ext acc = ge_identity();
        for (uint32_t e = lo + threadIdx.x; e < hi; e += blockDim.x) {
            uint32_t v = __ldg(slice + e), t = v & 0x7fffffffu;
            uint32_t pi = point_idx ? __ldg(point_idx + t) : (t | BP_POINT_DYNAMIC);
            const ge_niels *src = (pi & BP_POINT_DYNAMIC) ? pts_dynamic + (pi & 0x7fffffffu) : pts_static + pi;
            ge_niels q = ldg_niels(src);
            if (v & 0x80000000u) q = ge_niels_neg(q);
            acc = ge_madd(acc, q);
        }
#pragma unroll 1
        for (int d = 16; d >= 1; d >>= 1) { ge_ext o = shfl_down_ext(acc, d); acc = ge_add(acc, o); }
        if (lane == 0) sm[wid] = acc;
        __syncthreads();
        if (wid == 0) {
            ge_ext r = lane < (blockDim.x >> 5) ? sm[lane] : ge_identity();
#pragma unroll 1
            for (int d = 2; d >= 1; d >>= 1) { ge_ext o = shfl_down_ext(r, d); r = ge_add(r, o); }
            if (lane == 0) st_ext(buckets + gb, r);
        }
        __syncthreads();
    }
}
// pass 4: bucket accumulation, SPLIT adjacent lanes per bucket: each sums every SPLIT-th +-point of the bucket's slice (mixed
// additions), a shuffle tree adds the partial sums.  SPLIT > 1 trades (SPLIT-1) full additions per bucket for SPLIT x more warps
// in flight and a SPLIT x shorter serial chain per thread.
template <int SPLIT>
__global__ void __launch_bounds__(128, 5) k_msm_accumulate(const uint32_t *__restrict__ starts, const uint32_t *__restrict__ ends, const uint32_t *__restrict__ sorted,
                                                        const uint32_t *__restrict__ offsets, const uint32_t *__restrict__ order, int W, uint32_t nb, size_t n_buckets,
                                                        const uint32_t *__restrict__ point_idx, const ge_niels *__restrict__ pts_static, const ge_niels *__restrict__ pts_dynamic,
                                                        ge_ext *__restrict__ buckets, uint32_t heavy_min, uint32_t n_light_blocks, const uint32_t *__restrict__ heavy_n, const uint32_t *__restrict__ heavy) {
    const uint32_t n_heavy_blocks = gridDim.x - n_light_blocks;
    if (blockIdx.x < n_heavy_blocks) {        // the grid's FIRST blocks own the heavy buckets (listed by k_msm_order), one block per bucket: the longest work starts first
        msm_heavy_role(starts, ends, sorted, offsets, heavy_n, heavy, W, nb, point_idx, pts_static, pts_dynamic, buckets, blockIdx.x, n_heavy_blocks);
        return;
    }
    size_t tid = (size_t)(blockIdx.x - n_heavy_blocks) * blockDim.x + threadIdx.x;
    size_t b = tid / SPLIT; uint32_t sub = (uint32_t)(tid % SPLIT);
    bool live = b < n_buckets;
    if (SPLIT == 1 && !live) return;
    size_t gb = live ? order[b] : 0;
    size_t seg = gb / nb; uint32_t msm = (uint32_t)(seg / W), w = (uint32_t)(seg % W);
    uint32_t o0 = __ldg(offsets + msm), len = __ldg(offsets + msm + 1) - o0;
    const uint32_t *slice = sorted + msm_slice_base(o0, len, w, W);
    uint32_t lo = starts[gb], hi = ends[gb];
    if (hi - lo >= heavy_min) live = false;     // k_msm_accumulate_heavy owns this bucket
    if (!live) { if (SPLIT == 1) return; lo = hi = 0; }
    ge_ext acc = ge_identity();
    for (uint32_t e = lo + sub; e < hi; e += SPLIT) {
        uint32_t v = __ldg(slice + e), t = v & 0x7fffffffu;
        uint32_t pi = point_idx ? __ldg(point_idx + t) : (t | BP_POINT_DYNAMIC);
        const ge_niels *src = (pi & BP_POINT_DYNAMIC) ? pts_dynamic + (pi & 0x7fffffffu) : pts_static + pi;
        ge_niels q = ldg_niels(src);
        if (v & 0x80000000u) q = ge_niels_neg(q);
        acc = ge_madd(acc, q);
    }
    if (SPLIT > 1) {
#pragma unroll 1
        for (int d = SPLIT / 2; d >= 1; d >>= 1) { ge_ext o = shfl_down_ext(acc, d); acc = ge_add(acc, o); }
    }
    if (live && sub == 0) st_ext(buckets + gb, acc);
}
// pass 5: bucket reduction  R = sum_j (j+1) B_j  per segment, one block per segment.
// Each thread owns a contiguous chunk; a warp-shuffle suffix scan over the chunk sums gives every
// thread the sum of all buckets above its chunk, then one running-sum pass finishes the chunk and
// a shuffle tree adds the per-thread results.
__global__ void __launch_bounds__(256) k_msm_reduce(const ge_ext *__restrict__ buckets, uint32_t nb, ge_ext *__restrict__ window_sums) {
    __shared__ ge_ext sm[8];
    size_t seg = blockIdx.x;
    const ge_ext *B = buckets + seg * nb;
    uint32_t nthreads = blockDim.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nwarps = nthreads >> 5;
    uint32_t L = (nb + nthreads - 1) / nthreads;
    uint32_t lo = min(tid * L, nb), hi = min(lo + L, nb);
    // 1. chunk sum
    ge_ext S = ge_identity();
    for (uint32_t j = lo; j < hi; j++) S = ge_add(S, ld_ext(B + j));
    // 2. inclusive suffix scan across the block
    ge_ext suf = S;
#pragma unroll 1
    for (int d = 1; d < 32; d <<= 1) { ge_ext o = shfl_down_ext(suf, d); if (lane + d < 32) suf = ge_add(suf, o); }
    if (lane == 0) sm[wid] = suf;               // total of this warp
    __syncthreads();
    ge_ext above = ge_identity();               // total of the warps holding higher buckets
#pragma unroll 1
    for (uint32_t k = wid + 1; k < nwarps; k++) above = ge_add(above, sm[k]);
    // exclusive suffix: everything strictly above this thread's chunk
    ge_ext next = shfl_down_ext(suf, 1);
    ge_ext run = lane == 31 ? above : ge_add(next, above);
    // 3. running-sum pass over the chunk, top bucket first
    ge_ext acc = ge_identity();
    for (uint32_t j = hi; j > lo; j--) { run = ge_add(run, ld_ext(B + j - 1)); acc = ge_add(acc, run); }
    // 4. block sum of acc
#pragma unroll 1
    for (int d = 16; d >= 1; d >>= 1) { ge_ext o = shfl_down_ext(acc, d); acc = ge_add(acc, o); }
    __syncthreads();
    if (lane == 0) sm[wid] = acc;
    __syncthreads();
    if (tid == 0) { ge_ext r = sm[0]; for (uint32_t k = 1; k < nwarps; k++) r = ge_add(r, sm[k]); st_ext(window_sums + seg, r); }
}
// pass 6: window combination (Horner with c doublings per window), one thread per MSM
__global__ void k_msm_combine(const ge_ext *__restrict__ window_sums, uint32_t n_msm, int c, int W, ge_ext *__restrict__ results) {
    uint32_t m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n_msm) return;
    const ge_ext *R = window_sums + (size_t)m * W;
    ge_ext acc = ld_ext(R + W - 1);
#pragma unroll 1
    for (int w = W - 2; w >= 0; w--) {
#pragma unroll 1
        for (int i = 0; i < c; i++) acc = ge_dbl(acc);
        acc = ge_add(acc, ld_ext(R + w));
    }
    st_ext(results + m, acc);
}

// pass 6, latency-optimised form for few MSMs: four lanes per MSM, lane q holds coordinate q of the running point
// (X, Y, Z, T).  A doubling is then one squaring and one multiplication deep (the four squarings and the four products
// of the HWCD formulas run on the four lanes) plus two shuffle rounds, instead of eight field operations in sequence;
// the 253-doubling Horner chain is the longest dependency chain of a verified batch.
__device__ __forceinline__ fe shfl_fe4(const fe &v, int src) {
    fe r;
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = __shfl_sync(0xffffffffu, v.v[i], src, 4);
    return r;
}
__device__ __forceinline__ fe sel_fe(bool pick_b, const fe &a, const fe &b) { return fe_select(a, b, pick_b); }
__global__ void __launch_bounds__(32) k_msm_combine4(const ge_ext *__restrict__ window_sums, uint32_t n_msm, int c, int W, ge_ext *__restrict__ results) {
    uint32_t lane = threadIdx.x & 31, q = lane & 3;
    uint32_t m = blockIdx.x * 8 + (lane >> 2);
    bool active = m < n_msm;
    const ge_ext *R = window_sums + (size_t)(active ? m : n_msm - 1) * W;       // idle groups shadow the last MSM (shuffles need every lane)
    const fe d2 = fe_const_d2();
    fe cur = ld_fe(&R[W - 1].X + q);
#pragma unroll 1
    for (int w = W - 2; w >= 0; w--) {
#pragma unroll 1
        for (int i = 0; i < c; i++) {
            // doubling: A = X^2, B = Y^2, ZZ = Z^2, D = (X+Y)^2 on lanes 0..3
            fe x = shfl_fe4(cur, 0), y = shfl_fe4(cur, 1);
            fe sq = fe_sq(sel_fe(q == 3, cur, fe_add(x, y)));
            fe A = shfl_fe4(sq, 0), B = shfl_fe4(sq, 1), ZZ = shfl_fe4(sq, 2), D = shfl_fe4(sq, 3);
            fe H = fe_add(A, B), E = fe_sub(D, H), G = fe_sub(B, A), F = fe_sub(G, fe_dbl(ZZ)), Hn = fe_neg(H);
            // X3 = E F, Y3 = G Hn, Z3 = F G, T3 = E Hn
            fe o1 = sel_fe(q == 1, sel_fe(q == 2, E, F), G), o2 = sel_fe(q == 0, sel_fe(q == 2, Hn, G), F);
            cur = fe_mul(o1, o2);
        }
        // addition of the window sum (extended, from memory): lanes compute (Y1-X1)(Y2-X2), (Y1+X1)(Y2+X2), Z1 Z2, T1 (2d T2)
        const ge_ext *P2 = R + w;
        fe X2 = ld_fe(&P2->X), Y2 = ld_fe(&P2->Y), Z2 = ld_fe(&P2->Z), T2d = fe_mul(ld_fe(&P2->T), d2);
        fe x1 = shfl_fe4(cur, 0), y1 = shfl_fe4(cur, 1);
        fe a = sel_fe(q >= 2, sel_fe(q == 1, fe_sub(y1, x1), fe_add(y1, x1)), cur);
        fe b = sel_fe(q == 1, sel_fe(q == 2, sel_fe(q == 3, fe_sub(Y2, X2), T2d), Z2), fe_add(Y2, X2));
        fe pr = fe_mul(a, b);
        fe A = shfl_fe4(pr, 0), B = shfl_fe4(pr, 1), Dh = shfl_fe4(pr, 2), C = shfl_fe4(pr, 3);
        fe D = fe_dbl(Dh), E = fe_sub(B, A), F = fe_sub(D, C), G = fe_add(D, C), H = fe_add(B, A);
        // X3 = E F, Y3 = G H, Z3 = F G, T3 = E H
        fe o1 = sel_fe(q == 1, sel_fe(q == 2, E, F), G), o2 = sel_fe(q == 0, sel_fe(q == 2, H, G), F);
        cur = fe_mul(o1, o2);
    }
    if (active) st_fe(&results[m].X + q, cur);
}

// ------------------------------------------------------------------ K4: IPP generator fold
// out[i] = s_lo[i] * P[i] + s_hi[i] * P[half + i], written back to P[i] in affine Niels form
// (InnerProductProof::create's G/H fold, /root/reference/src/inner_product_proof.rs:127-134,177-178).
// One thread per i: joint double-and-add over the two scalars (shared doublings), then one inversion
// to renormalise so that the next round's MSMs keep using 7-multiplication mixed additions.
// scalars: canonical 32-byte little-endian; stride 0 = the same pair for every i (later rounds).
__global__ void __launch_bounds__(64) k_ipp_fold(ge_niels *__restrict__ P, uint32_t half, const uint8_t *__restrict__ s_lo, const uint8_t *__restrict__ s_hi, uint32_t stride) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= half) return;
    uint8_t b1[32], b2[32]; ld32(b1, s_lo + (size_t)i * stride); ld32(b2, s_hi + (size_t)i * stride);
    sc k1 = sc_load(b1), k2 = sc_load(b2);
    ge_niels p1 = ldg_niels(P + i), p2 = ldg_niels(P + half + i);
    ge_ext e12 = ge_madd(ge_from_niels(p1), p2);
    fe zi = fe_invert(e12.Z);
    ge_niels p12 = ge_to_niels_affine(fe_mul(e12.X, zi), fe_mul(e12.Y, zi));
    ge_ext acc = ge_identity();
#pragma unroll 1
    for (int bit = 252; bit >= 0; bit--) {
        acc = ge_dbl(acc);
        uint32_t d = ((k1.v[bit >> 5] >> (bit & 31)) & 1u) | (((k2.v[bit >> 5] >> (bit & 31)) & 1u) << 1);
        if (d) { ge_niels q = d == 1 ? p1 : (d == 2 ? p2 : p12); acc = ge_madd(acc, q); }
    }
    fe zf = fe_invert(acc.Z);
    st_niels(P + i, ge_to_niels_affine(fe_mul(acc.X, zf), fe_mul(acc.Y, zf)));
}
// ------------------------------------------------------------------ K4': inner-product prover without generator folding
// InnerProductProof::create (inner_product_proof.rs:69-185) folds G and H every round (N two-term scalar multiplications in total).
// The device session never folds points: after rounds with challenges u_1..u_j the folded generator at position i is the combination
//   G^(j)[i] = sum over original indices idx = i (mod n_j) of cG[idx] G[idx],   cG[idx] = G_factors[idx] * prod_r u_r^(+-1)
// (sign by the index bit the round consumed; H likewise with the signs swapped), so L_j and R_j are MSMs of N + 1 terms over the
// ORIGINAL resident points with scalars a_L[pos - h] * cG[idx] etc.; a round costs O(N) scalar products and one MSM launch chain.
// a, b are kept in Montgomery form, the coefficient vectors cG, cH in plain form, so that every product needed as an MSM scalar comes
// out of one Montgomery multiplication as a canonical value.  B proofs of the same length run side by side.
struct ippx_geom { uint32_t N, B, n; };        // N = original length, n = current length (power of two), B proofs
__global__ void __launch_bounds__(128) k_ippx_init(ippx_geom g, const uint8_t *__restrict__ a_in, const uint8_t *__restrict__ b_in, const uint8_t *__restrict__ Gf, const uint8_t *__restrict__ Hf,
                                                   sc *__restrict__ a, sc *__restrict__ b, sc *__restrict__ cG, sc *__restrict__ cH) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)g.B * g.N) return;
    a[i] = sc_to_mont(sc_load(a_in + 32 * i)); b[i] = sc_to_mont(sc_load(b_in + 32 * i));
    sc one = sc_zero(); one.v[0] = 1;
    cG[i] = Gf ? sc_load(Gf + 32 * i) : one; cH[i] = Hf ? sc_load(Hf + 32 * i) : one;
}
// c_L = <a_L, b_R>, c_R = <a_R, b_L> (inner_product_proof.rs:84-85,150-151): block (proof, which), canonical bytes into slot N of the proof's L / R scalar row
__global__ void __launch_bounds__(128) k_ippx_inner(ippx_geom g, const sc *__restrict__ a, const sc *__restrict__ b, uint8_t *__restrict__ scal) {
    __shared__ sc sm[4];
    const uint32_t p = blockIdx.x >> 1, which = blockIdx.x & 1, h = g.n >> 1;
    const sc *x = a + (size_t)p * g.N + (which ? h : 0), *y = b + (size_t)p * g.N + (which ? 0 : h);
    sc acc = sc_zero();
    for (uint32_t i0 = threadIdx.x * 16; i0 < h; i0 += blockDim.x * 16) {      // 16 products per lazy reduction
        sc_wide w = sc_wide_zero();
        for (uint32_t i = i0; i < min(i0 + 16, h); i++) sc_wide_mac(w, x[i], y[i]);
        acc = sc_add(acc, sc_wide_redc(w));
    }
    for (int d = 16; d >= 1; d >>= 1) { sc o; for (int i = 0; i < 8; i++) o.v[i] = __shfl_down_sync(0xffffffffu, acc.v[i], d); acc = sc_add(acc, o); }
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (uint32_t k = 1; k < (blockDim.x >> 5); k++) acc = sc_add(acc, sm[k]);
        uint8_t bytes[32]; sc_store(bytes, sc_from_mont(acc)); st32(scal + (((size_t)p * 2 + which) * (g.N + 1) + g.N) * 32, bytes);
    }
}
// MSM rows of the round: per proof an L row and an R row of N + 1 (scalar, point index) pairs.  gidx/hidx = table slots of the original G / H
// points, Q = dynamic point p.
__global__ void __launch_bounds__(128) k_ippx_rows(ippx_geom g, const sc *__restrict__ a, const sc *__restrict__ b, const sc *__restrict__ cG, const sc *__restrict__ cH,
                                                   const uint32_t *__restrict__ gidx, const uint32_t *__restrict__ hidx, uint8_t *__restrict__ scal, uint32_t *__restrict__ pidx) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (size_t)g.B * g.N) return;
    const uint32_t p = (uint32_t)(t / g.N), idx = (uint32_t)(t % g.N), h = g.n >> 1, pos = idx & (g.n - 1), blk = idx / g.n;
    const sc *ap = a + (size_t)p * g.N, *bp_ = b + (size_t)p * g.N;
    const size_t rowL = ((size_t)p * 2) * (g.N + 1), rowR = rowL + g.N + 1;
    uint8_t bytes[32];
    // G[idx]: right half -> L with a_L, left half -> R with a_R (inner_product_proof.rs:87-99,101-113)
    { bool right = pos >= h; uint32_t i = right ? pos - h : pos;
      sc v = sc_mont_mul(right ? ap[i] : ap[h + i], cG[t]);
      size_t slot = (right ? rowL : rowR) + blk * h + i;
      sc_store(bytes, v); st32(scal + slot * 32, bytes); pidx[slot] = gidx[idx]; }
    // H[idx]: left half -> L with b_R, right half -> R with b_L
    { bool left = pos < h; uint32_t i = left ? pos : pos - h;
      sc v = sc_mont_mul(left ? bp_[h + i] : bp_[i], cH[t]);
      size_t slot = (left ? rowL : rowR) + (g.N >> 1) + blk * h + i;
      sc_store(bytes, v); st32(scal + slot * 32, bytes); pidx[slot] = hidx[idx]; }
    if (idx == 0) { pidx[rowL + g.N] = BP_POINT_DYNAMIC | p; pidx[rowR + g.N] = BP_POINT_DYNAMIC | p; }
}
// apply the round's challenge: a' = a_L u + u^-1 a_R, b' = b_L u^-1 + u b_R (:125-126,175-176); cG *= u^-1 (left) / u (right), cH *= u / u^-1 (:127-134,177-178)
__global__ void __launch_bounds__(128) k_ippx_fold(ippx_geom g, const uint8_t *__restrict__ u_bytes, const uint8_t *__restrict__ uinv_bytes, sc *__restrict__ a, sc *__restrict__ b,
                                                   sc *__restrict__ cG, sc *__restrict__ cH) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (size_t)g.B * g.N) return;
    const uint32_t p = (uint32_t)(t / g.N), idx = (uint32_t)(t % g.N), h = g.n >> 1, pos = idx & (g.n - 1);
    const sc u = sc_to_mont(sc_load(u_bytes + 32 * p)), ui = sc_to_mont(sc_load(uinv_bytes + 32 * p));
    cG[t] = sc_mont_mul(cG[t], pos < h ? ui : u);
    cH[t] = sc_mont_mul(cH[t], pos < h ? u : ui);
    if (idx < h) {
        sc *ap = a + (size_t)p * g.N, *bp_ = b + (size_t)p * g.N;
        ap[idx] = sc_add(sc_mont_mul(ap[idx], u), sc_mont_mul(ui, ap[h + idx]));
        bp_[idx] = sc_add(sc_mont_mul(bp_[idx], ui), sc_mont_mul(u, bp_[h + idx]));
    }
}
__global__ void k_ippx_final(ippx_geom g, const sc *__restrict__ a, const sc *__restrict__ b, uint8_t *__restrict__ out) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= g.B) return;
    uint8_t bytes[32];
    sc_store(bytes, sc_from_mont(a[(size_t)p * g.N])); st32(out + 64 * p, bytes);
    sc_store(bytes, sc_from_mont(b[(size_t)p * g.N])); st32(out + 64 * p + 32, bytes);
}

// ------------------------------------------------------------------ range-proof batch verification kernels
// One launch group verifies `nbatch` independent batches of `count` proofs each: every batch has its own random-linear-
// combination MSM of T = S + count*D terms and its own accept flag; the per-proof kernels run over all nbatch*count proofs.
struct rp_geom { uint32_t n, m, k, N, D, S; uint32_t proof_len; uint32_t count, nbatch, T; };   // D = 4+2k+m dynamic terms, S = 2+2N static terms

// Per-call parameter block, uploaded through a pinned staging ring; kernels read the input addresses from it so that the
// launch sequence itself is the same for every call on a reserved geometry (captured once as a CUDA graph).
struct rp_params {
    uint8_t tstate[208];                       // serialized transcript (BP_TRANSCRIPT_BYTES used)
    uint8_t seed[32];                          // external randomness of the batching weights
    const uint8_t *proofs, *commitments;       // device addresses: nbatch*count proofs / nbatch*count*m commitments
    uint32_t *verdict;                         // device address: nbatch*count verdict codes
    uint8_t pad_[512 - 208 - 32 - 24];
};
static_assert(sizeof(rp_params) == 512, "parameter block");

__device__ __forceinline__ uint32_t rp_eff_status(uint32_t st, uint32_t dec_bad) {          // an undecodable point is a VerificationError (mod.rs:445)
    return st != BP_PROOF_OK ? st : (dec_bad ? (uint32_t)BP_PROOF_VERIFICATION_ERROR : (uint32_t)BP_PROOF_OK);
}

// K6: transcript replay (pure hashing).  One thread per proof (32 proofs per warp, identical control flow, every lane busy); the STROBE
// state of each thread is a padded shared-memory row (stride 204 B: conflict-free byte access).  The proof bytes are read straight from
// global memory: staging the block's 32 proofs (21 KB) in shared memory through the TMA engine was built and measured -- same solo
// duration (the kernel is bound by its ~22 Keccak-f per proof, not by the byte loads) and 4 % less throughput for the whole mix, because
// 29 KB of shared memory per 32-thread block changes what can be co-resident on an SM (profiles/r2_experiments.md).
#define RP_TR_THREADS 32
__global__ void __launch_bounds__(RP_TR_THREADS) k_rp_transcript(const rp_params *__restrict__ par, rp_geom g, uint32_t total,
                                                                   uint8_t *__restrict__ raw, uint32_t *__restrict__ status) {
    __shared__ __align__(16) uint8_t rows[RP_TR_THREADS][204];
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= total) return;
    const uint8_t *proof = par->proofs + (size_t)p * g.proof_len, *V = par->commitments + (size_t)p * g.m * 32;
    uint8_t (*my)[64] = reinterpret_cast<uint8_t (*)[64]>(raw + (size_t)p * (RP_RAW_U + g.k) * 64);
    status[p] = rp_transcript_raw(my, proof, g.k, V, g.n, g.m, par->tstate, par->seed, rows[threadIdx.x]);
}
// Lean head: ONE thread per proof runs the sequential statement (rp_scalars_head) -- ~180 dependent Montgomery products.  Several
// groups are in flight, so a head's latency is hidden; what counts is its footprint: one warp per 32 proofs here against eight
// (a 256-thread block at 100 registers per 32 proofs = two thirds of the GPU's register file for a whole group) in the round-1 cooperative head.
__global__ void __launch_bounds__(32) k_rp_head_seq(const rp_params *__restrict__ par, rp_geom g, const uint8_t *__restrict__ raw, uint32_t total,
                                                    rp_head *__restrict__ heads, sc *__restrict__ tabs, const sc *__restrict__ pow2, uint32_t *__restrict__ status) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= total) return;
    rp_head &h = heads[p];
    uint32_t st = status[p];
    if (st != BP_PROOF_OK) { h.status = st; return; }
    const uint8_t *rw = raw + (size_t)p * (RP_RAW_U + g.k) * 64;
    rp_challenges ch;
    ch.y = rp_wide(rw + 64 * RP_RAW_Y); ch.z = rp_wide(rw + 64 * RP_RAW_Z); ch.x = rp_wide(rw + 64 * RP_RAW_X); ch.w = rp_wide(rw + 64 * RP_RAW_W);
    ch.c = rp_wide(rw + 64 * RP_RAW_C); ch.rho = rp_wide(rw + 64 * RP_RAW_RHO);
    bool bad = sc_is_zero(ch.y);
    for (uint32_t j = 0; j < g.k; j++) { ch.u[j] = rp_wide(rw + 64 * (RP_RAW_U + j)); bad = bad || sc_is_zero(ch.u[j]); }
    if (bad) { status[p] = BP_PROOF_VERIFICATION_ERROR; h.status = BP_PROOF_VERIFICATION_ERROR; return; }      // zero challenge: see rp_transcript
    if (sc_is_zero(ch.rho)) ch.rho = sc_mont_one();
    rp_scalars_head(h, tabs + (size_t)p * rp_tab_size(g.k, g.m), pow2, ch, par->proofs + (size_t)p * g.proof_len, g.k, g.n, g.m);
    h.status = BP_PROOF_OK;
}
// K5 (combined check): verification scalars with the sum over the proofs taken in registers.  Block = (chunk of RP_CHUNK proofs of one
// batch); thread = generator index i: it walks the chunk's proofs and adds up their weighted g_i and h_i (three Montgomery products
// per proof and index), so the count x S per-proof array of the per-proof form below is never written; k_rp_static_sum then adds
// the few per-chunk partial sums.  The same block also writes the chunk's per-proof ("dynamic") scalars into the MSM scalar array.
#define RP_CHUNK 32
__global__ void __launch_bounds__(128) k_rp_scalars_sum(rp_geom g, const rp_head *__restrict__ heads, const sc *__restrict__ tabs, const uint32_t *__restrict__ dec_bad,
                                                        sc *__restrict__ part, uint8_t *__restrict__ scal) {
    __shared__ uint32_t okmask;
    const uint32_t nchunks = (g.count + RP_CHUNK - 1) / RP_CHUNK, b = blockIdx.x / nchunks, ch = blockIdx.x % nchunks;
    const uint32_t q0 = ch * RP_CHUNK, nq = min((uint32_t)RP_CHUNK, g.count - q0), p0 = b * g.count + q0;
    if (threadIdx.x < 32) {
        bool ok = threadIdx.x < nq && heads[p0 + threadIdx.x].status == BP_PROOF_OK && !dec_bad[p0 + threadIdx.x];
        uint32_t m_ = __ballot_sync(0xffffffffu, ok);
        if (threadIdx.x == 0) okmask = m_;
    }
    __syncthreads();
    const uint32_t mask = okmask, tsz = rp_tab_size(g.k, g.m);
    sc *mine = part + ((size_t)b * nchunks + ch) * g.S;
    // weighted g_i = -zL - A_hi[hi] s_lo[lo],  h_i = zL + P_hi[hi] P_lo[lo] - Q_hi[hi] Q_lo[lo]  (rp_scalars_gh): the three products of the
    // chunk's proofs are summed as 512-bit integers and reduced once per chunk (RP_CHUNK <= 32 products fit), one third of the multiplies
    const uint32_t kl = rp_kl(g.k), TL = 1u << kl;
    for (uint32_t i = threadIdx.x; i < g.N; i += blockDim.x) {
        const uint32_t lo = i & (TL - 1), hi = i >> kl;
        sc zsum = sc_zero();
        sc_wide accA = sc_wide_zero(), accP = sc_wide_zero(), accQ = sc_wide_zero();
        for (uint32_t q = 0; q < nq; q++) {
            if (!((mask >> q) & 1u)) continue;
            rp_tabs T = rp_tab_ptrs(const_cast<sc *>(tabs) + (size_t)(p0 + q) * tsz, g.k);
            zsum = sc_add(zsum, heads[p0 + q].zL);
            sc_wide_mac(accA, T.A_hi[hi], T.s_lo[lo]); sc_wide_mac(accP, T.P_hi[hi], T.P_lo[lo]); sc_wide_mac(accQ, T.Q_hi[hi], T.Q_lo[lo]);
        }
        mine[2 + i] = sc_sub(sc_neg(zsum), sc_wide_redc(accA));
        mine[2 + g.N + i] = sc_sub(sc_add(zsum, sc_wide_redc(accP)), sc_wide_redc(accQ));
    }
    if (threadIdx.x < 2) {
        sc s0 = sc_zero();
        for (uint32_t q = 0; q < nq; q++) if ((mask >> q) & 1u) s0 = sc_add(s0, threadIdx.x == 0 ? heads[p0 + q].blinding_scalar : heads[p0 + q].basepoint_scalar);
        mine[threadIdx.x] = s0;
    }
    for (uint32_t e = threadIdx.x; e < nq * g.D; e += blockDim.x) {
        uint32_t q = e / g.D, d = e % g.D;
        sc v = ((mask >> q) & 1u) ? sc_from_mont(rp_scalars_dynamic(heads[p0 + q], d, g.k)) : sc_zero();
        uint8_t bytes[32]; sc_store(bytes, v); st32(scal + ((size_t)b * g.T + g.S + (size_t)(q0 + q) * g.D + d) * 32, bytes);
    }
}
// add the per-chunk partial sums of a batch's static-term scalars: one warp per (static term, batch)
__global__ void __launch_bounds__(32) k_rp_static_sum(const sc *__restrict__ part, rp_geom g, uint8_t *__restrict__ scal) {
    const uint32_t nchunks = (g.count + RP_CHUNK - 1) / RP_CHUNK, s = blockIdx.x, b = blockIdx.y;
    sc acc = sc_zero();
    for (uint32_t c = threadIdx.x; c < nchunks; c += 32) acc = sc_add(acc, part[((size_t)b * nchunks + c) * g.S + s]);
    for (int d = 16; d >= 1; d >>= 1) {
        sc o; for (int i = 0; i < 8; i++) o.v[i] = __shfl_down_sync(0xffffffffu, acc.v[i], d);
        acc = sc_add(acc, o);
    }
    if (threadIdx.x == 0) { uint8_t bytes[32]; sc_store(bytes, sc_from_mont(acc)); st32(scal + ((size_t)b * g.T + s) * 32, bytes); }
}
// K5 (per-proof form, used by the fallback): one thread per (proof, term) with term in
// [0, N) -> (g_i, h_i) and [N, N + D) -> the per-proof scalars.
//   contrib : total x S Montgomery scalars (weighted static-term scalars: B~, B, G.., H..)
//   scal    : nbatch x T canonical scalars, the MSM scalar arrays; the D scalars of proof q of batch b start at b*T + S + q*D
// A proof that is malformed or has an undecodable point contributes nothing to its batch's combination.
__global__ void __launch_bounds__(128) k_rp_scalars(rp_geom g, const rp_head *__restrict__ heads, const sc *__restrict__ tabs, const uint32_t *__restrict__ dec_bad,
                                                    uint32_t total, sc *__restrict__ contrib, uint8_t *__restrict__ scal) {
    uint32_t per = g.N + g.D;
    size_t gi = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gi >= (size_t)total * per) return;
    uint32_t p = (uint32_t)(gi / per), i = (uint32_t)(gi % per);
    const rp_head &h = heads[p];
    sc *my = contrib + (size_t)p * g.S;
    bool ok = h.status == BP_PROOF_OK && !dec_bad[p];
    if (i < g.N) {
        sc gg = sc_zero(), hh = sc_zero();
        if (ok) rp_scalars_gh(h, tabs + (size_t)p * rp_tab_size(g.k, g.m), i, g.k, gg, hh);
        my[2 + i] = gg; my[2 + g.N + i] = hh;
        if (i == 0) { my[0] = ok ? h.blinding_scalar : sc_zero(); my[1] = ok ? h.basepoint_scalar : sc_zero(); }
    } else {
        uint32_t d = i - g.N, b = p / g.count, q = p % g.count;
        sc v = ok ? sc_from_mont(rp_scalars_dynamic(h, d, g.k)) : sc_zero();
        uint8_t bytes[32]; sc_store(bytes, v); st32(scal + ((size_t)b * g.T + g.S + (size_t)q * g.D + d) * 32, bytes);
    }
}
// decompress the per-proof points in MSM order A,S,T_1,T_2,L..,R..,V.. straight out of the proof bytes; independent of the
// transcript, so it runs beside k_rp_transcript / k_rp_head_seq (second branch of the launch graph).  The proofs and commitments a
// block's 128 points come from are contiguous: they are staged with two TMA bulk copies, the 32-byte encodings are read from shared memory.
#define RP_DEC_THREADS 128
__global__ void __launch_bounds__(RP_DEC_THREADS, 5) k_rp_decompress(const rp_params *__restrict__ par, rp_geom g, uint32_t total,
                                                                  ge_niels *__restrict__ out, uint32_t *__restrict__ dec_bad) {
    extern __shared__ __align__(128) uint8_t dec_smem[];
    __shared__ __align__(8) uint64_t bar;
    const size_t i0 = (size_t)blockIdx.x * blockDim.x, i = i0 + threadIdx.x, n_pts = (size_t)total * g.D;
    const uint32_t pf = (uint32_t)(i0 / g.D), pl = (uint32_t)((min(i0 + blockDim.x, n_pts) - 1) / g.D), np = pl - pf + 1;     // proofs this block touches
    uint8_t *sp = dec_smem, *sv = dec_smem + (size_t)(RP_DEC_THREADS / g.D + 2) * g.proof_len;
    tma_stage_two(sp, par->proofs + (size_t)pf * g.proof_len, np * g.proof_len, sv, par->commitments + (size_t)pf * g.m * 32, np * g.m * 32, &bar);
    if (i >= n_pts) return;
    uint32_t p = (uint32_t)(i / g.D), idx = (uint32_t)(i % g.D);
    const uint8_t *proof = sp + (size_t)(p - pf) * g.proof_len, *src;
    if (idx < 4) src = proof + 32 * idx;
    else if (idx < 4 + g.k) src = proof + 224 + 64 * (idx - 4);
    else if (idx < 4 + 2 * g.k) src = proof + 224 + 64 * (idx - 4 - g.k) + 32;
    else src = sv + ((size_t)(p - pf) * g.m + (idx - 4 - 2 * g.k)) * 32;
    uint8_t s[32]; lds32(s, src);
    fe x, y; bool valid = ge_decode(x, y, s);
    st_niels(out + i, valid ? ge_to_niels_affine(x, y) : ge_niels_identity());
    if (!valid) dec_bad[p] = 1u;
}
// fallback, first level: one combined MSM per chunk of RP_CHUNK proofs of a failing batch.  Everything is already there: the chunk's
// summed static-term scalars (k_rp_scalars_sum's partial sums) and its proofs' dynamic scalars.  Rows are [S static | RP_CHUNK*D dynamic],
// the tail of a short last chunk padded with zero scalars (a zero scalar never touches its point).
__global__ void k_rp_chunk_rows(const sc *__restrict__ part_b, const uint8_t *__restrict__ dyn_b, rp_geom g, uint32_t gens_cap, uint32_t gens_parties, uint32_t dyn_base,
                                uint8_t *__restrict__ out_scalars, uint32_t *__restrict__ out_pidx) {
    const uint32_t nchunks = (g.count + RP_CHUNK - 1) / RP_CHUNK, row = g.S + RP_CHUNK * g.D;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)nchunks * row) return;
    uint32_t ch = (uint32_t)(i / row), t = (uint32_t)(i % row);
    uint8_t b[32]; uint32_t v;
    if (t < g.S) {
        sc_store(b, sc_from_mont(part_b[(size_t)ch * g.S + t]));
        if (t < 2) v = t;
        else if (t < 2 + g.N) { uint32_t q = t - 2; v = gens_slot(0u, q / g.n, q % g.n, gens_cap, gens_parties); }
        else { uint32_t q = t - 2 - g.N; v = gens_slot(1u, q / g.n, q % g.n, gens_cap, gens_parties); }
    } else {
        uint32_t e = t - g.S, q = ch * RP_CHUNK + e / g.D;
        if (q < g.count) { ld32(b, dyn_b + ((size_t)q * g.D + e % g.D) * 32); v = BP_POINT_DYNAMIC | (dyn_base + q * g.D + e % g.D); }
        else { for (int j = 0; j < 32; j++) b[j] = 0; v = 0; }
    }
    st32(out_scalars + 32 * i, b); out_pidx[i] = v;
}
// verdicts of the proofs in chunks whose combined check passed (the failing chunks are re-checked proof by proof); chunk_ok[ch] = identity flags
__global__ void k_rp_verdict_chunks(const uint32_t *__restrict__ status, const uint32_t *__restrict__ dec_bad, const ge_ext *__restrict__ results, uint32_t count,
                                    uint32_t *__restrict__ verdict, uint32_t *__restrict__ chunk_ok) {
    uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= count) return;
    uint32_t ch = q / RP_CHUNK;
    bool ok = ge_is_identity(ld_ext(results + ch));
    if (q % RP_CHUNK == 0) chunk_ok[ch] = ok ? 1u : 0u;
    if (ok) verdict[q] = rp_eff_status(status[q], dec_bad[q]);
}
// fallback: expand contrib (Montgomery) into per-proof canonical scalar rows [S static | D dynamic] for the proofs of one batch;
// contrib / dyn_scalars point at the batch's first proof
__global__ void k_rp_expand_scalars(const sc *__restrict__ contrib, const uint8_t *__restrict__ dyn_scalars, rp_geom g, uint32_t count, uint8_t *__restrict__ out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t row = g.S + g.D;
    if (i >= (size_t)count * row) return;
    uint32_t p = (uint32_t)(i / row), t = (uint32_t)(i % row);
    uint8_t b[32];
    if (t < g.S) sc_store(b, sc_from_mont(contrib[(size_t)p * g.S + t]));
    else ld32(b, dyn_scalars + ((size_t)p * g.D + (t - g.S)) * 32);
    st32(out + 32 * i, b);
}
// final verdicts of the combined check, one block per batch: the batch's MSM result must lie in the identity coset
// (mod.rs:447); every well-formed proof inherits that result, malformed ones keep their own code; batch_ok[b] = all accepted
__global__ void __launch_bounds__(256) k_rp_verdict_batch(const uint32_t *__restrict__ status, const uint32_t *__restrict__ dec_bad, const ge_ext *__restrict__ results,
                                                          rp_geom g, const rp_params *__restrict__ par, uint32_t *__restrict__ batch_ok, uint32_t *__restrict__ combined_ok) {
    __shared__ uint32_t s_ok, s_all;
    uint32_t b = blockIdx.x;
    if (threadIdx.x == 0) { s_ok = ge_is_identity(ld_ext(results + b)) ? 1u : 0u; s_all = 1u; }
    __syncthreads();
    uint32_t ok = s_ok, all = 1u;
    uint32_t *verdict = par->verdict;
    for (uint32_t q = threadIdx.x; q < g.count; q += blockDim.x) {
        uint32_t p = b * g.count + q;
        uint32_t st = rp_eff_status(status[p], dec_bad[p]);
        uint32_t v = st != BP_PROOF_OK ? st : (ok ? (uint32_t)BP_PROOF_OK : (uint32_t)BP_PROOF_VERIFICATION_ERROR);
        verdict[p] = v;
        if (v != BP_PROOF_OK) all = 0u;
    }
    if (!all) atomicExch(&s_all, 0u);
    __syncthreads();
    if (threadIdx.x == 0) { batch_ok[b] = s_all; combined_ok[b] = s_ok; }       // combined_ok = 0: the per-proof recheck has to find the offenders
}
// per-proof verdicts after the fallback MSMs (one result per proof); arrays point at the batch's first proof
__global__ void k_rp_verdict_proofs(const uint32_t *__restrict__ status, const uint32_t *__restrict__ dec_bad, const ge_ext *__restrict__ results, uint32_t count,
                                    uint32_t *__restrict__ verdict) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= count) return;
    uint32_t st = rp_eff_status(status[p], dec_bad[p]);
    verdict[p] = st != BP_PROOF_OK ? st : (ge_is_identity(ld_ext(results + p)) ? (uint32_t)BP_PROOF_OK : (uint32_t)BP_PROOF_VERIFICATION_ERROR);
}

// ------------------------------------------------------------------ constant-time indexed MSM (msm_ct.cuh, bp_msm_indexed_batch_ct)
// recode: one thread per term.  digits: T x 64 signed bytes; msm_err bit 1 = a non-canonical scalar in that MSM (the atomic is issued
// for every term, with the flag as its operand, so neither its address nor its presence depends on the scalar)
__global__ void __launch_bounds__(128) k_msm_ct_recode(const uint8_t *__restrict__ scalars, const uint32_t *__restrict__ offsets, uint32_t n_msm, uint32_t T,
                                                       int8_t *__restrict__ digits, uint32_t *__restrict__ msm_err) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    const uint4 *p = reinterpret_cast<const uint4 *>(scalars + 32 * (size_t)t);
    uint4 a = p[0], b = p[1];
    uint32_t s[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    uint32_t bad = ct_scalar_geq_l_mask(s);
    for (int i = 0; i < 8; i++) s[i] &= ~bad;                        // a rejected scalar contributes nothing
    uint32_t d[CT_DIGITS];
    ct_recode_radix16(s, d);
    uint32_t w[CT_DIGITS / 4];
#pragma unroll
    for (int i = 0; i < CT_DIGITS / 4; i++) w[i] = (d[4 * i] & 0xffu) | ((d[4 * i + 1] & 0xffu) << 8) | ((d[4 * i + 2] & 0xffu) << 16) | ((d[4 * i + 3] & 0xffu) << 24);
    uint4 *o = reinterpret_cast<uint4 *>(digits + (size_t)CT_DIGITS * t);
#pragma unroll
    for (int i = 0; i < CT_DIGITS / 16; i++) o[i] = make_uint4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
    uint32_t msm = n_msm == 1 ? 0u : msm_of_term(offsets, n_msm, t);
    atomicOr(msm_err + msm, bad & 2u);
}

// table: one thread per term, [1..8]P of table slot point_idx[t] (public data only)
__global__ void __launch_bounds__(128) k_msm_ct_table(const uint32_t *__restrict__ point_idx, uint32_t T, const ge_niels *__restrict__ gens, ge_ext *__restrict__ tab) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    ge_ext *o = tab + (size_t)CT_TABLE * t;
    ct_table(ge_from_niels(ldg_niels(gens + __ldg(point_idx + t))), [&](int j, const ge_ext &p) { st_ext(o + j, p); });
}

// straus: one thread per chunk [chunks[c], chunks[c+1]) of consecutive terms of one MSM
__global__ void __launch_bounds__(128) k_msm_ct_straus(const uint32_t *__restrict__ chunks, uint32_t n_chunks, const int8_t *__restrict__ digits,
                                                       const ge_ext *__restrict__ tab, ge_ext *__restrict__ partial) {
    uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_chunks) return;
    const uint32_t lo = __ldg(chunks + c), hi = __ldg(chunks + c + 1);
    ge_ext acc = ge_identity();
#pragma unroll 1
    for (int w = CT_DIGITS - 1; w >= 0; w--) {
        if (w != CT_DIGITS - 1) {
#pragma unroll 1
            for (int i = 0; i < 4; i++) acc = ge_dbl(acc);
        }
#pragma unroll 1
        for (uint32_t t = lo; t < hi; t++) {
            const uint32_t d = (uint32_t)(int32_t)__ldg(digits + (size_t)CT_DIGITS * t + w);
            const uint32_t *base = reinterpret_cast<const uint32_t *>(tab + (size_t)CT_TABLE * t);
            ge_ext e = ct_lookup(d, [&](uint32_t j, int k, uint32_t *v) { uint4 x = __ldg(reinterpret_cast<const uint4 *>(base + 32 * j + k)); v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w; });
            acc = ge_add(acc, e);
        }
    }
    st_ext(partial + c, acc);
}

// reduce: one block per MSM; thread i adds chunks i, i + blockDim, ... of the MSM, then a shuffle tree and one shared-memory round
#define CT_REDUCE_THREADS 128
__global__ void __launch_bounds__(CT_REDUCE_THREADS) k_msm_ct_reduce(const ge_ext *__restrict__ partial, const uint32_t *__restrict__ msm_chunks, ge_ext *__restrict__ results) {
    __shared__ ge_ext sm[CT_REDUCE_THREADS / 32];
    const uint32_t m = blockIdx.x, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const uint32_t c0 = __ldg(msm_chunks + m), c1 = __ldg(msm_chunks + m + 1);
    ge_ext acc = ge_identity();
#pragma unroll 1
    for (uint32_t c = c0 + threadIdx.x; c < c1; c += blockDim.x) acc = ge_add(acc, ld_ext(partial + c));
#pragma unroll 1
    for (int d = 16; d >= 1; d >>= 1) { ge_ext o = shfl_down_ext(acc, d); acc = ge_add(acc, o); }
    if (lane == 0) sm[wid] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        ge_ext r = sm[0];
#pragma unroll 1
        for (uint32_t k = 1; k < CT_REDUCE_THREADS / 32; k++) r = ge_add(r, sm[k]);
        st_ext(results + m, r);
    }
}
