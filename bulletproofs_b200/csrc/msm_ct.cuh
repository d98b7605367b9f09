// Constant-time multiscalar multiplication over generator-table slots (bp_msm_indexed_batch_ct).
//
// The reference computes every commitment that holds a prover secret with curve25519-dalek's constant-time Straus
// (RistrettoPoint::multiscalar_mul: signed radix-16 digits, a lookup table of [1..8]P per term read in full and combined with
// masks).  This is the same algorithm on the device.  Public, and free to steer control flow and addresses: term counts, the
// MSM offsets, the point indices (table slots) and the output point.  Secret: the scalars.  Nothing below branches on a scalar,
// indexes memory with one, or lets one choose a launch; the only scalar-derived value that leaves the kernels is the per-MSM
// canonicality verdict.
//
//   recode : per term, canonicality as a mask (a non-canonical scalar is zeroed, its MSM flagged), then 64 signed digits in [-8, 8]
//            with the carries done arithmetically
//   table  : per term, [1..8]P in extended coordinates from the resident table entry (public data only)
//   straus : one thread per chunk of consecutive terms of one MSM (chunks are cut from the offsets alone): 64 windows of four shared
//            doublings, then per term one masked selection over all eight entries and one complete addition
//   reduce : the chunk partials of each MSM in a fixed tree (k_compress then encodes the public result)
// The kernels are in kernels.cuh (k_msm_ct_*); this header holds what they share with the host-side tests.
//
// The recoding and the selection are templates on their word type W.  The product instantiates them with uint32_t; the CPU test
// tier instantiates them a second time with a wrapper type that has arithmetic and bitwise operators but no conversion to bool or
// to an integer, so that a branch or an index on a scalar-derived value fails to compile there (tests/host_emul/ct_audit.cpp).
// The group operations they feed (ge_add, ge_dbl, fe_cneg_mask) are fixed carry chains and multiplier rows with no data-dependent
// control flow (fe.cuh).
#pragma once
#include "ge.cuh"
#include "sc.cuh"

#define CT_DIGITS 64                 // signed radix-16 digits of a scalar < 2^253
#define CT_TABLE 8                   // [1..8]P per term

// all-ones when a == b, else zero (no comparison instruction on the secret: the top bit of x | -x is set iff x != 0)
template <class W> BP_HD W ct_mask_eq(const W &a, uint32_t b) {
    W x = a ^ b;
    return ((x | (~x + 1u)) >> 31) - 1u;
}

// all-ones when the 256-bit little-endian value s >= l, else zero: the borrow out of s - l, computed word by word without a compare
template <class W> BP_HD W ct_scalar_geq_l_mask(const W s[8]) {
    const uint32_t L[8] = SC_L_LIMBS;
    W borrow = s[0] ^ s[0];          // zero of type W
    for (int i = 0; i < 8; i++) {
        W d = s[i] - L[i] - borrow;
        borrow = ((~s[i] & L[i]) | (~(s[i] ^ L[i]) & d)) >> 31;
    }
    return borrow - 1u;              // borrow = 1 <=> s < l
}

// s (canonical, < l < 2^253) -> 64 signed digits d[i] in [-8, 8] (two's complement words), sum d[i] 16^i = s.  Nibble i is read with
// public shifts; the carry into digit i+1 is (nibble + carry + 8) >> 4.  The top digit absorbs the last carry: nibble 63 of a value
// below 2^253 is at most 1, so d[63] <= 2.
template <class W> BP_HD void ct_recode_radix16(const W s[8], W d[CT_DIGITS]) {
    W carry = s[0] ^ s[0];
    for (int i = 0; i < CT_DIGITS - 1; i++) {
        W v = ((s[i >> 3] >> (4 * (i & 7))) & 15u) + carry;
        carry = (v + 8u) >> 4;
        d[i] = v - (carry << 4);
    }
    d[CT_DIGITS - 1] = ((s[7] >> 28) & 15u) + carry;
}

// sign mask (all-ones for a negative digit) and absolute value of a two's-complement digit
template <class W> BP_HD void ct_digit_split(const W &d, W &neg, W &abs) {
    neg = ~(d >> 31) + 1u;
    abs = (d ^ neg) - neg;
}

// out = entry |d| of the term's table, or the identity for d = 0: every one of the eight entries is loaded and merged under a mask.
// load4(j, k, q) reads words k..k+3 of entry j (public addresses).  Point words: X[0..8) Y[8..16) Z[16..24) T[24..32).
template <class W, class Load4> BP_HD void ct_select_entry(const W &abs, Load4 load4, W out[32]) {
    for (int k = 0; k < 32; k++) out[k] = abs ^ abs;
    out[8] = out[8] + 1u; out[16] = out[16] + 1u;                   // identity (0 : 1 : 1 : 0)
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (uint32_t j = 0; j < CT_TABLE; j++) {
        W m = ct_mask_eq(abs, j + 1);
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (int k = 0; k < 32; k += 4) {
            uint32_t q[4]; load4(j, k, q);
            for (int i = 0; i < 4; i++) out[k + i] = out[k + i] ^ ((out[k + i] ^ q[i]) & m);
        }
    }
}

// [1..8]P from P (public): store(j, point) receives (j + 1) P for j = 0..7
template <class Store> BP_HD void ct_table(const ge_ext &p1, Store store) {
    ge_ext p2 = ge_dbl(p1), p4 = ge_dbl(p2);
    store(0, p1); store(1, p2); store(3, p4);
    ge_ext p3 = ge_add(p2, p1); store(2, p3);
    store(4, ge_add(p4, p1));
    ge_ext p6 = ge_dbl(p3); store(5, p6);
    store(6, ge_add(p6, p1));
    store(7, ge_dbl(p4));
}

// d P for a signed digit d in [-8, 8] (two's-complement word) from the term's table: all eight entries read, -P = (-X : Y : Z : -T) by mask
template <class Load4> BP_HD ge_ext ct_lookup(uint32_t d, Load4 load4) {
    uint32_t neg, abs, q[32];
    ct_digit_split(d, neg, abs);
    ct_select_entry(abs, load4, q);
    ge_ext e;
    for (int i = 0; i < 8; i++) { e.X.v[i] = q[i]; e.Y.v[i] = q[8 + i]; e.Z.v[i] = q[16 + i]; e.T.v[i] = q[24 + i]; }
    e.X = fe_cneg_mask(e.X, neg); e.T = fe_cneg_mask(e.T, neg);
    return e;
}
