// Field arithmetic mod p = 2^255 - 19 for sm_100a.
//
// Representation: eight saturated 32-bit limbs, value v in [0, 2^256) taken mod p ("weakly
// reduced": any representative below 2^256 is allowed between operations; 2^256 = 38 mod p).
// This replaces the 5x51-bit-limb u64 backend the reference gets from curve25519-dalek
// (/root/reference/Cargo.toml:21).  Why not 51-bit limbs on the GPU: the integer pipe multiplies
// 32x32->64 (IMAD.WIDE); a 51-bit limb product costs four of those plus carries, so radix 2^32
// needs 64+8 wide multiplies per field product where radix 2^51 needs ~100+ (DESIGN.md §fe).
//
// All multi-instruction asm blocks mark their pure outputs early-clobber ("=&r"): an output is written
// before the last input is read, so it must never share a register with a (dying) input.
//
// Every function is __host__ __device__: under __CUDA_ARCH__ the hot operations are PTX
// carry chains (mad.lo.cc / madc.hi.cc pairs, which ptxas fuses into IMAD.WIDE.U32.X); on the
// host a portable 64-bit-accumulator version of the same limb algorithm is compiled so that
// tests/host_emul can unit-test all device math on the CPU box.  The host path is test-only:
// nothing in the product library calls it.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define BP_HD __host__ __device__ __forceinline__
#define BP_HDN __host__ __device__ __noinline__
#else
#define BP_HD inline
#define BP_HDN inline
#endif

struct fe { uint32_t v[8]; };

BP_HD fe fe_zero() { fe r; for (int i = 0; i < 8; i++) r.v[i] = 0; return r; }
BP_HD fe fe_one() { fe r = fe_zero(); r.v[0] = 1; return r; }
BP_HD fe fe_small(uint32_t x) { fe r = fe_zero(); r.v[0] = x; return r; }

// r = a + b
BP_HD fe fe_add(const fe &a, const fe &b) {
    fe r;
#ifdef __CUDA_ARCH__
    uint32_t c;
    asm("add.cc.u32 %0, %9, %17;\n\t"
        "addc.cc.u32 %1, %10, %18;\n\t"
        "addc.cc.u32 %2, %11, %19;\n\t"
        "addc.cc.u32 %3, %12, %20;\n\t"
        "addc.cc.u32 %4, %13, %21;\n\t"
        "addc.cc.u32 %5, %14, %22;\n\t"
        "addc.cc.u32 %6, %15, %23;\n\t"
        "addc.cc.u32 %7, %16, %24;\n\t"
        "addc.u32 %8, 0, 0;\n\t"
        : "=&r"(r.v[0]), "=&r"(r.v[1]), "=&r"(r.v[2]), "=&r"(r.v[3]), "=&r"(r.v[4]), "=&r"(r.v[5]), "=&r"(r.v[6]), "=&r"(r.v[7]), "=&r"(c)
        : "r"(a.v[0]), "r"(a.v[1]), "r"(a.v[2]), "r"(a.v[3]), "r"(a.v[4]), "r"(a.v[5]), "r"(a.v[6]), "r"(a.v[7]),
          "r"(b.v[0]), "r"(b.v[1]), "r"(b.v[2]), "r"(b.v[3]), "r"(b.v[4]), "r"(b.v[5]), "r"(b.v[6]), "r"(b.v[7]));
    // fold the carry: 2^256 = 38.  A second carry can only happen when the wrapped value is tiny.
    uint32_t k = c * 38u, c2;
    asm("add.cc.u32 %0, %0, %9;\n\t"
        "addc.cc.u32 %1, %1, 0;\n\t"
        "addc.cc.u32 %2, %2, 0;\n\t"
        "addc.cc.u32 %3, %3, 0;\n\t"
        "addc.cc.u32 %4, %4, 0;\n\t"
        "addc.cc.u32 %5, %5, 0;\n\t"
        "addc.cc.u32 %6, %6, 0;\n\t"
        "addc.cc.u32 %7, %7, 0;\n\t"
        "addc.u32 %8, 0, 0;\n\t"
        : "+r"(r.v[0]), "+r"(r.v[1]), "+r"(r.v[2]), "+r"(r.v[3]), "+r"(r.v[4]), "+r"(r.v[5]), "+r"(r.v[6]), "+r"(r.v[7]), "=&r"(c2)
        : "r"(k));
    r.v[0] += c2 * 38u;
#else
    uint64_t c = 0;
    for (int i = 0; i < 8; i++) { c += (uint64_t)a.v[i] + b.v[i]; r.v[i] = (uint32_t)c; c >>= 32; }
    uint64_t k = c * 38;
    for (int i = 0; i < 8; i++) { k += r.v[i]; r.v[i] = (uint32_t)k; k >>= 32; }
    r.v[0] += (uint32_t)k * 38u;
#endif
    return r;
}

// r = a - b
BP_HD fe fe_sub(const fe &a, const fe &b) {
    fe r;
#ifdef __CUDA_ARCH__
    uint32_t bw;
    asm("sub.cc.u32 %0, %9, %17;\n\t"
        "subc.cc.u32 %1, %10, %18;\n\t"
        "subc.cc.u32 %2, %11, %19;\n\t"
        "subc.cc.u32 %3, %12, %20;\n\t"
        "subc.cc.u32 %4, %13, %21;\n\t"
        "subc.cc.u32 %5, %14, %22;\n\t"
        "subc.cc.u32 %6, %15, %23;\n\t"
        "subc.cc.u32 %7, %16, %24;\n\t"
        "subc.u32 %8, 0, 0;\n\t"
        : "=&r"(r.v[0]), "=&r"(r.v[1]), "=&r"(r.v[2]), "=&r"(r.v[3]), "=&r"(r.v[4]), "=&r"(r.v[5]), "=&r"(r.v[6]), "=&r"(r.v[7]), "=&r"(bw)
        : "r"(a.v[0]), "r"(a.v[1]), "r"(a.v[2]), "r"(a.v[3]), "r"(a.v[4]), "r"(a.v[5]), "r"(a.v[6]), "r"(a.v[7]),
          "r"(b.v[0]), "r"(b.v[1]), "r"(b.v[2]), "r"(b.v[3]), "r"(b.v[4]), "r"(b.v[5]), "r"(b.v[6]), "r"(b.v[7]));
    // bw = 0 or 0xffffffff.  A borrow means the true value is r - 2^256 = r - 38 (mod p).
    uint32_t k = bw & 38u, b2;
    asm("sub.cc.u32 %0, %0, %9;\n\t"
        "subc.cc.u32 %1, %1, 0;\n\t"
        "subc.cc.u32 %2, %2, 0;\n\t"
        "subc.cc.u32 %3, %3, 0;\n\t"
        "subc.cc.u32 %4, %4, 0;\n\t"
        "subc.cc.u32 %5, %5, 0;\n\t"
        "subc.cc.u32 %6, %6, 0;\n\t"
        "subc.cc.u32 %7, %7, 0;\n\t"
        "subc.u32 %8, 0, 0;\n\t"
        : "+r"(r.v[0]), "+r"(r.v[1]), "+r"(r.v[2]), "+r"(r.v[3]), "+r"(r.v[4]), "+r"(r.v[5]), "+r"(r.v[6]), "+r"(r.v[7]), "=&r"(b2)
        : "r"(k));
    r.v[0] -= b2 & 38u;
#else
    int64_t c = 0;
    for (int i = 0; i < 8; i++) { c += (int64_t)a.v[i] - b.v[i]; r.v[i] = (uint32_t)c; c >>= 32; }
    int64_t k = c * 38;   // c = 0 or -1
    for (int i = 0; i < 8; i++) { k += r.v[i]; r.v[i] = (uint32_t)k; k >>= 32; }
    r.v[0] += (uint32_t)(k * 38);
#endif
    return r;
}

BP_HD fe fe_neg(const fe &a) { return fe_sub(fe_zero(), a); }

#ifdef __CUDA_ARCH__
// acc[0..7] (+)= a[j0], a[j0+2], a[j0+4], a[j0+6] times b, 64-bit products tiled over acc; returns carry-out
#define BP_MULROW(e0, e1, e2, e3, e4, e5, e6, e7, a0, a2, a4, a6, bi)                                   \
    asm("mul.lo.u32 %0, %8, %12;\n\t mul.hi.u32 %1, %8, %12;\n\t"                                      \
        "mul.lo.u32 %2, %9, %12;\n\t mul.hi.u32 %3, %9, %12;\n\t"                                      \
        "mul.lo.u32 %4, %10, %12;\n\t mul.hi.u32 %5, %10, %12;\n\t"                                    \
        "mul.lo.u32 %6, %11, %12;\n\t mul.hi.u32 %7, %11, %12;\n\t"                                    \
        : "=&r"(e0), "=&r"(e1), "=&r"(e2), "=&r"(e3), "=&r"(e4), "=&r"(e5), "=&r"(e6), "=&r"(e7)              \
        : "r"(a0), "r"(a2), "r"(a4), "r"(a6), "r"(bi))
// chain add of four products into eight existing limbs, carry-out into `co` (fresh limb)
#define BP_MADROW(e0, e1, e2, e3, e4, e5, e6, e7, co, a0, a2, a4, a6, bi)                               \
    asm("mad.lo.cc.u32 %0, %9, %13, %0;\n\t madc.hi.cc.u32 %1, %9, %13, %1;\n\t"                       \
        "madc.lo.cc.u32 %2, %10, %13, %2;\n\t madc.hi.cc.u32 %3, %10, %13, %3;\n\t"                    \
        "madc.lo.cc.u32 %4, %11, %13, %4;\n\t madc.hi.cc.u32 %5, %11, %13, %5;\n\t"                    \
        "madc.lo.cc.u32 %6, %12, %13, %6;\n\t madc.hi.cc.u32 %7, %12, %13, %7;\n\t"                    \
        "addc.u32 %8, 0, 0;\n\t"                                                                        \
        : "+r"(e0), "+r"(e1), "+r"(e2), "+r"(e3), "+r"(e4), "+r"(e5), "+r"(e6), "+r"(e7), "=&r"(co)    \
        : "r"(a0), "r"(a2), "r"(a4), "r"(a6), "r"(bi))
// same, but carry-out is added into an existing small limb `co`
#define BP_MADROW_ACC(e0, e1, e2, e3, e4, e5, e6, e7, co, a0, a2, a4, a6, bi)                           \
    asm("mad.lo.cc.u32 %0, %9, %13, %0;\n\t madc.hi.cc.u32 %1, %9, %13, %1;\n\t"                       \
        "madc.lo.cc.u32 %2, %10, %13, %2;\n\t madc.hi.cc.u32 %3, %10, %13, %3;\n\t"                    \
        "madc.lo.cc.u32 %4, %11, %13, %4;\n\t madc.hi.cc.u32 %5, %11, %13, %5;\n\t"                    \
        "madc.lo.cc.u32 %6, %12, %13, %6;\n\t madc.hi.cc.u32 %7, %12, %13, %7;\n\t"                    \
        "addc.u32 %8, %8, 0;\n\t"                                                                       \
        : "+r"(e0), "+r"(e1), "+r"(e2), "+r"(e3), "+r"(e4), "+r"(e5), "+r"(e6), "+r"(e7), "+r"(co)    \
        : "r"(a0), "r"(a2), "r"(a4), "r"(a6), "r"(bi))
// the top two limbs are fresh (zero): six existing limbs, then a product written with carry-in; carry-out to fresh `co`
#define BP_MADROW_EXT(e0, e1, e2, e3, e4, e5, e6, e7, co, a0, a2, a4, a6, bi)                           \
    asm("mad.lo.cc.u32 %0, %9, %13, %0;\n\t madc.hi.cc.u32 %1, %9, %13, %1;\n\t"                       \
        "madc.lo.cc.u32 %2, %10, %13, %2;\n\t madc.hi.cc.u32 %3, %10, %13, %3;\n\t"                    \
        "madc.lo.cc.u32 %4, %11, %13, %4;\n\t madc.hi.cc.u32 %5, %11, %13, %5;\n\t"                    \
        "madc.lo.cc.u32 %6, %12, %13, %6;\n\t madc.hi.cc.u32 %7, %12, %13, 0;\n\t"                     \
        "addc.u32 %8, 0, 0;\n\t"                                                                        \
        : "+r"(e0), "+r"(e1), "+r"(e2), "+r"(e3), "+r"(e4), "+r"(e5), "+r"(e6), "=&r"(e7), "=&r"(co)    \
        : "r"(a0), "r"(a2), "r"(a4), "r"(a6), "r"(bi))
#endif

// 16-limb product t = a*b
BP_HD void fe_mul_wide(uint32_t t[16], const fe &A, const fe &B) {
#ifdef __CUDA_ARCH__
    const uint32_t *a = A.v, *b = B.v;
    // even-aligned accumulator e[0..15] and odd-aligned accumulator o[0..14] (value o << 32);
    // row i adds a_j*b_i to e if i+j is even, to o otherwise (see DESIGN.md §fe for the limb ranges)
    uint32_t e0, e1, e2, e3, e4, e5, e6, e7, e8, e9, e10, e11, e12, e13, e14, e15;
    uint32_t o0, o1, o2, o3, o4, o5, o6, o7, o8, o9, o10, o11, o12, o13, o14;
    // row 0: e[0..7] = a0,a2,a4,a6 * b0 ; o[0..7] = a1,a3,a5,a7 * b0
    BP_MULROW(e0, e1, e2, e3, e4, e5, e6, e7, a[0], a[2], a[4], a[6], b[0]);
    BP_MULROW(o0, o1, o2, o3, o4, o5, o6, o7, a[1], a[3], a[5], a[7], b[0]);
    // row 1: o[0..7] += a0,a2,a4,a6 * b1 -> o8 ; e[2..9] += a1,a3,a5,a7 * b1 (e8,e9 fresh) -> e10
    BP_MADROW(o0, o1, o2, o3, o4, o5, o6, o7, o8, a[0], a[2], a[4], a[6], b[1]);
    e8 = 0;
    BP_MADROW_EXT(e2, e3, e4, e5, e6, e7, e8, e9, e10, a[1], a[3], a[5], a[7], b[1]);
    // row 2: e[2..9] += a0,a2,a4,a6 * b2 -> e10 += ; o[2..9] += a1,a3,a5,a7 * b2 (o9 fresh) -> o10
    BP_MADROW_ACC(e2, e3, e4, e5, e6, e7, e8, e9, e10, a[0], a[2], a[4], a[6], b[2]);
    BP_MADROW_EXT(o2, o3, o4, o5, o6, o7, o8, o9, o10, a[1], a[3], a[5], a[7], b[2]);
    // row 3: o[2..9] += a0.. * b3 -> o10 += ; e[4..11] += a1.. * b3 (e11 fresh) -> e12
    BP_MADROW_ACC(o2, o3, o4, o5, o6, o7, o8, o9, o10, a[0], a[2], a[4], a[6], b[3]);
    BP_MADROW_EXT(e4, e5, e6, e7, e8, e9, e10, e11, e12, a[1], a[3], a[5], a[7], b[3]);
    // row 4
    BP_MADROW_ACC(e4, e5, e6, e7, e8, e9, e10, e11, e12, a[0], a[2], a[4], a[6], b[4]);
    BP_MADROW_EXT(o4, o5, o6, o7, o8, o9, o10, o11, o12, a[1], a[3], a[5], a[7], b[4]);
    // row 5
    BP_MADROW_ACC(o4, o5, o6, o7, o8, o9, o10, o11, o12, a[0], a[2], a[4], a[6], b[5]);
    BP_MADROW_EXT(e6, e7, e8, e9, e10, e11, e12, e13, e14, a[1], a[3], a[5], a[7], b[5]);
    // row 6
    BP_MADROW_ACC(e6, e7, e8, e9, e10, e11, e12, e13, e14, a[0], a[2], a[4], a[6], b[6]);
    BP_MADROW_EXT(o6, o7, o8, o9, o10, o11, o12, o13, o14, a[1], a[3], a[5], a[7], b[6]);
    // row 7: o[6..13] += a0.. * b7 -> o14 += ; e[8..15] += a1.. * b7 (e15 fresh), no carry out (product < 2^512)
    BP_MADROW_ACC(o6, o7, o8, o9, o10, o11, o12, o13, o14, a[0], a[2], a[4], a[6], b[7]);
    uint32_t dead;
    BP_MADROW_EXT(e8, e9, e10, e11, e12, e13, e14, e15, dead, a[1], a[3], a[5], a[7], b[7]);
    (void)dead;
    // t = e + (o << 32)
    t[0] = e0;
    asm("add.cc.u32 %0, %15, %30;\n\t"
        "addc.cc.u32 %1, %16, %31;\n\t"
        "addc.cc.u32 %2, %17, %32;\n\t"
        "addc.cc.u32 %3, %18, %33;\n\t"
        "addc.cc.u32 %4, %19, %34;\n\t"
        "addc.cc.u32 %5, %20, %35;\n\t"
        "addc.cc.u32 %6, %21, %36;\n\t"
        "addc.cc.u32 %7, %22, %37;\n\t"
        "addc.cc.u32 %8, %23, %38;\n\t"
        "addc.cc.u32 %9, %24, %39;\n\t"
        "addc.cc.u32 %10, %25, %40;\n\t"
        "addc.cc.u32 %11, %26, %41;\n\t"
        "addc.cc.u32 %12, %27, %42;\n\t"
        "addc.cc.u32 %13, %28, %43;\n\t"
        "addc.u32 %14, %29, %44;\n\t"
        : "=&r"(t[1]), "=&r"(t[2]), "=&r"(t[3]), "=&r"(t[4]), "=&r"(t[5]), "=&r"(t[6]), "=&r"(t[7]), "=&r"(t[8]),
          "=&r"(t[9]), "=&r"(t[10]), "=&r"(t[11]), "=&r"(t[12]), "=&r"(t[13]), "=&r"(t[14]), "=&r"(t[15])
        : "r"(e1), "r"(e2), "r"(e3), "r"(e4), "r"(e5), "r"(e6), "r"(e7), "r"(e8), "r"(e9), "r"(e10), "r"(e11), "r"(e12), "r"(e13), "r"(e14), "r"(e15),
          "r"(o0), "r"(o1), "r"(o2), "r"(o3), "r"(o4), "r"(o5), "r"(o6), "r"(o7), "r"(o8), "r"(o9), "r"(o10), "r"(o11), "r"(o12), "r"(o13), "r"(o14));
#else
    uint64_t acc[16];
    for (int i = 0; i < 16; i++) acc[i] = 0;
    // column sums split in low/high halves so nothing overflows 64 bits
    for (int i = 0; i < 8; i++)
        for (int j = 0; j < 8; j++) {
            uint64_t p = (uint64_t)A.v[i] * B.v[j];
            acc[i + j] += (uint32_t)p;
            acc[i + j + 1] += p >> 32;
        }
    uint64_t c = 0;
    for (int i = 0; i < 16; i++) { c += acc[i]; t[i] = (uint32_t)c; c >>= 32; }
#endif
}

// r = (t[0..7] + 38 * t[8..15]) folded below 2^256
BP_HD fe fe_reduce_wide(const uint32_t t[16]) {
    fe r;
#ifdef __CUDA_ARCH__
    uint32_t r0 = t[0], r1 = t[1], r2 = t[2], r3 = t[3], r4 = t[4], r5 = t[5], r6 = t[6], r7 = t[7], ce;
    uint32_t u0, u1, u2, u3, u4, u5, u6, u7;
    const uint32_t k38 = 38u;
    // even-aligned: (r0,r1) += t8*38, (r2,r3) += t10*38, ... carry -> ce
    BP_MADROW(r0, r1, r2, r3, r4, r5, r6, r7, ce, t[8], t[10], t[12], t[14], k38);
    // odd-aligned: u[0..7] = t9*38, t11*38, t13*38, t15*38 at limbs 1..8
    BP_MULROW(u0, u1, u2, u3, u4, u5, u6, u7, t[9], t[11], t[13], t[15], k38);
    uint32_t c8;
    asm("add.cc.u32 %0, %0, %8;\n\t"
        "addc.cc.u32 %1, %1, %9;\n\t"
        "addc.cc.u32 %2, %2, %10;\n\t"
        "addc.cc.u32 %3, %3, %11;\n\t"
        "addc.cc.u32 %4, %4, %12;\n\t"
        "addc.cc.u32 %5, %5, %13;\n\t"
        "addc.cc.u32 %6, %6, %14;\n\t"
        "addc.u32 %7, %15, %16;\n\t"
        : "+r"(r1), "+r"(r2), "+r"(r3), "+r"(r4), "+r"(r5), "+r"(r6), "+r"(r7), "=&r"(c8)
        : "r"(u0), "r"(u1), "r"(u2), "r"(u3), "r"(u4), "r"(u5), "r"(u6), "r"(u7), "r"(ce));
    // c8 <= 39: fold once more, then a last conditional +38
    uint32_t k = c8 * 38u, c2;
    asm("add.cc.u32 %0, %0, %9;\n\t"
        "addc.cc.u32 %1, %1, 0;\n\t"
        "addc.cc.u32 %2, %2, 0;\n\t"
        "addc.cc.u32 %3, %3, 0;\n\t"
        "addc.cc.u32 %4, %4, 0;\n\t"
        "addc.cc.u32 %5, %5, 0;\n\t"
        "addc.cc.u32 %6, %6, 0;\n\t"
        "addc.cc.u32 %7, %7, 0;\n\t"
        "addc.u32 %8, 0, 0;\n\t"
        : "+r"(r0), "+r"(r1), "+r"(r2), "+r"(r3), "+r"(r4), "+r"(r5), "+r"(r6), "+r"(r7), "=&r"(c2)
        : "r"(k));
    r0 += c2 * 38u;
    r.v[0] = r0; r.v[1] = r1; r.v[2] = r2; r.v[3] = r3; r.v[4] = r4; r.v[5] = r5; r.v[6] = r6; r.v[7] = r7;
#else
    uint64_t c = 0;
    for (int i = 0; i < 8; i++) { c += (uint64_t)t[i] + (uint64_t)t[i + 8] * 38u; r.v[i] = (uint32_t)c; c >>= 32; }
    uint64_t k = c * 38;                     // c <= 38
    for (int i = 0; i < 8; i++) { k += r.v[i]; r.v[i] = (uint32_t)k; k >>= 32; }
    r.v[0] += (uint32_t)k * 38u;
#endif
    return r;
}

// -DBP_NOINLINE_MUL: out-of-line multiplier (5x faster compile, 3x smaller kernels, ~7 % slower verification on B200:
// the field elements then travel through local memory) -- for debug builds only
#ifdef BP_NOINLINE_MUL
#define BP_FEMUL BP_HDN
#else
#define BP_FEMUL BP_HD
#endif
BP_FEMUL fe fe_mul(const fe &a, const fe &b) { uint32_t t[16]; fe_mul_wide(t, a, b); return fe_reduce_wide(t); }
// 16-limb square t = a*a: 28 off-diagonal products (each used once, then doubled) + 8 diagonal ones
BP_HD void fe_sq_wide(uint32_t t[16], const fe &A) {
#ifdef __CUDA_ARCH__
    const uint32_t *a = A.v;
    // S = sum_{i<j} a_i a_j 2^(32(i+j)) in an even-aligned (e[2..13]) and an odd-aligned (o[0..13], value o << 32)
    // accumulator, row by row as in fe_mul_wide; the limb ranges are derived in DESIGN.md §fe
    uint32_t e2, e3, e4, e5, e6, e7, e8, e9, e10, e11, e12, e13;
    uint32_t o0, o1, o2, o3, o4, o5, o6, o7, o8, o9, o10, o11, o12, o13;
    // row 0: e[2..7] = (a2,a4,a6)*a0 ; o[0..7] = (a1,a3,a5,a7)*a0
    asm("mul.lo.u32 %0, %6, %9;\n\t mul.hi.u32 %1, %6, %9;\n\t"
        "mul.lo.u32 %2, %7, %9;\n\t mul.hi.u32 %3, %7, %9;\n\t"
        "mul.lo.u32 %4, %8, %9;\n\t mul.hi.u32 %5, %8, %9;\n\t"
        : "=&r"(e2), "=&r"(e3), "=&r"(e4), "=&r"(e5), "=&r"(e6), "=&r"(e7) : "r"(a[2]), "r"(a[4]), "r"(a[6]), "r"(a[0]));
    BP_MULROW(o0, o1, o2, o3, o4, o5, o6, o7, a[1], a[3], a[5], a[7], a[0]);
    // row 1: o[2..7] += (a2,a4,a6)*a1 -> o8 ; e[4..7] += (a3,a5)*a1, (e8,e9) = a7*a1 + carry -> e10
    asm("mad.lo.cc.u32 %0, %7, %10, %0;\n\t madc.hi.cc.u32 %1, %7, %10, %1;\n\t"
        "madc.lo.cc.u32 %2, %8, %10, %2;\n\t madc.hi.cc.u32 %3, %8, %10, %3;\n\t"
        "madc.lo.cc.u32 %4, %9, %10, %4;\n\t madc.hi.cc.u32 %5, %9, %10, %5;\n\t"
        "addc.u32 %6, 0, 0;\n\t"
        : "+r"(o2), "+r"(o3), "+r"(o4), "+r"(o5), "+r"(o6), "+r"(o7), "=&r"(o8) : "r"(a[2]), "r"(a[4]), "r"(a[6]), "r"(a[1]));
    asm("mad.lo.cc.u32 %0, %7, %10, %0;\n\t madc.hi.cc.u32 %1, %7, %10, %1;\n\t"
        "madc.lo.cc.u32 %2, %8, %10, %2;\n\t madc.hi.cc.u32 %3, %8, %10, %3;\n\t"
        "madc.lo.cc.u32 %4, %9, %10, 0;\n\t madc.hi.cc.u32 %5, %9, %10, 0;\n\t"
        "addc.u32 %6, 0, 0;\n\t"
        : "+r"(e4), "+r"(e5), "+r"(e6), "+r"(e7), "=&r"(e8), "=&r"(e9), "=&r"(e10) : "r"(a[3]), "r"(a[5]), "r"(a[7]), "r"(a[1]));
    // row 2: o[4..7] += (a3,a5)*a2, (o8,o9) = a7*a2 + o8 -> o10 ; e[6..9] += (a4,a6)*a2 -> e10 +=
    asm("mad.lo.cc.u32 %0, %7, %10, %0;\n\t madc.hi.cc.u32 %1, %7, %10, %1;\n\t"
        "madc.lo.cc.u32 %2, %8, %10, %2;\n\t madc.hi.cc.u32 %3, %8, %10, %3;\n\t"
        "madc.lo.cc.u32 %4, %9, %10, %4;\n\t madc.hi.cc.u32 %5, %9, %10, 0;\n\t"
        "addc.u32 %6, 0, 0;\n\t"
        : "+r"(o4), "+r"(o5), "+r"(o6), "+r"(o7), "+r"(o8), "=&r"(o9), "=&r"(o10) : "r"(a[3]), "r"(a[5]), "r"(a[7]), "r"(a[2]));
    asm("mad.lo.cc.u32 %0, %5, %7, %0;\n\t madc.hi.cc.u32 %1, %5, %7, %1;\n\t"
        "madc.lo.cc.u32 %2, %6, %7, %2;\n\t madc.hi.cc.u32 %3, %6, %7, %3;\n\t"
        "addc.u32 %4, %4, 0;\n\t"
        : "+r"(e6), "+r"(e7), "+r"(e8), "+r"(e9), "+r"(e10) : "r"(a[4]), "r"(a[6]), "r"(a[2]));
    // row 3: o[6..9] += (a4,a6)*a3 -> o10 += ; (e8,e9) += a5*a3, (e10,e11) = a7*a3 + e10 -> e12
    asm("mad.lo.cc.u32 %0, %5, %7, %0;\n\t madc.hi.cc.u32 %1, %5, %7, %1;\n\t"
        "madc.lo.cc.u32 %2, %6, %7, %2;\n\t madc.hi.cc.u32 %3, %6, %7, %3;\n\t"
        "addc.u32 %4, %4, 0;\n\t"
        : "+r"(o6), "+r"(o7), "+r"(o8), "+r"(o9), "+r"(o10) : "r"(a[4]), "r"(a[6]), "r"(a[3]));
    asm("mad.lo.cc.u32 %0, %5, %7, %0;\n\t madc.hi.cc.u32 %1, %5, %7, %1;\n\t"
        "madc.lo.cc.u32 %2, %6, %7, %2;\n\t madc.hi.cc.u32 %3, %6, %7, 0;\n\t"
        "addc.u32 %4, 0, 0;\n\t"
        : "+r"(e8), "+r"(e9), "+r"(e10), "=&r"(e11), "=&r"(e12) : "r"(a[5]), "r"(a[7]), "r"(a[3]));
    // row 4: (o8,o9) += a5*a4, (o10,o11) = a7*a4 + o10 -> o12 ; (e10,e11) += a6*a4 -> e12 +=
    asm("mad.lo.cc.u32 %0, %5, %7, %0;\n\t madc.hi.cc.u32 %1, %5, %7, %1;\n\t"
        "madc.lo.cc.u32 %2, %6, %7, %2;\n\t madc.hi.cc.u32 %3, %6, %7, 0;\n\t"
        "addc.u32 %4, 0, 0;\n\t"
        : "+r"(o8), "+r"(o9), "+r"(o10), "=&r"(o11), "=&r"(o12) : "r"(a[5]), "r"(a[7]), "r"(a[4]));
    asm("mad.lo.cc.u32 %0, %3, %4, %0;\n\t madc.hi.cc.u32 %1, %3, %4, %1;\n\t addc.u32 %2, %2, 0;\n\t"
        : "+r"(e10), "+r"(e11), "+r"(e12) : "r"(a[6]), "r"(a[4]));
    // row 5: (o10,o11) += a6*a5 -> o12 += ; (e12,e13) = a7*a5 + e12
    asm("mad.lo.cc.u32 %0, %3, %4, %0;\n\t madc.hi.cc.u32 %1, %3, %4, %1;\n\t addc.u32 %2, %2, 0;\n\t"
        : "+r"(o10), "+r"(o11), "+r"(o12) : "r"(a[6]), "r"(a[5]));
    asm("mad.lo.cc.u32 %0, %2, %3, %0;\n\t madc.hi.u32 %1, %2, %3, 0;\n\t" : "+r"(e12), "=&r"(e13) : "r"(a[7]), "r"(a[5]));
    // row 6: (o12,o13) = a7*a6 + o12
    asm("mad.lo.cc.u32 %0, %2, %3, %0;\n\t madc.hi.u32 %1, %2, %3, 0;\n\t" : "+r"(o12), "=&r"(o13) : "r"(a[7]), "r"(a[6]));
    // S = e + (o << 32): S1 = o0, S_p = e_p + o_(p-1) for p = 2..13, S14 = o13 + carry, S15 = carry
    uint32_t s2, s3, s4, s5, s6, s7, s8, s9, s10, s11, s12, s13, s14, s15;
    asm("add.cc.u32 %0, %14, %26;\n\t"
        "addc.cc.u32 %1, %15, %27;\n\t"
        "addc.cc.u32 %2, %16, %28;\n\t"
        "addc.cc.u32 %3, %17, %29;\n\t"
        "addc.cc.u32 %4, %18, %30;\n\t"
        "addc.cc.u32 %5, %19, %31;\n\t"
        "addc.cc.u32 %6, %20, %32;\n\t"
        "addc.cc.u32 %7, %21, %33;\n\t"
        "addc.cc.u32 %8, %22, %34;\n\t"
        "addc.cc.u32 %9, %23, %35;\n\t"
        "addc.cc.u32 %10, %24, %36;\n\t"
        "addc.cc.u32 %11, %25, %37;\n\t"
        "addc.cc.u32 %12, %38, 0;\n\t"
        "addc.u32 %13, 0, 0;\n\t"
        : "=&r"(s2), "=&r"(s3), "=&r"(s4), "=&r"(s5), "=&r"(s6), "=&r"(s7), "=&r"(s8), "=&r"(s9), "=&r"(s10), "=&r"(s11), "=&r"(s12), "=&r"(s13), "=&r"(s14), "=&r"(s15)
        : "r"(e2), "r"(e3), "r"(e4), "r"(e5), "r"(e6), "r"(e7), "r"(e8), "r"(e9), "r"(e10), "r"(e11), "r"(e12), "r"(e13),
          "r"(o1), "r"(o2), "r"(o3), "r"(o4), "r"(o5), "r"(o6), "r"(o7), "r"(o8), "r"(o9), "r"(o10), "r"(o11), "r"(o12), "r"(o13));
    // x = 2S (limbs 1..15)
    uint32_t x1, x2, x3, x4, x5, x6, x7, x8, x9, x10, x11, x12, x13, x14, x15;
    asm("add.cc.u32 %0, %15, %15;\n\t"
        "addc.cc.u32 %1, %16, %16;\n\t"
        "addc.cc.u32 %2, %17, %17;\n\t"
        "addc.cc.u32 %3, %18, %18;\n\t"
        "addc.cc.u32 %4, %19, %19;\n\t"
        "addc.cc.u32 %5, %20, %20;\n\t"
        "addc.cc.u32 %6, %21, %21;\n\t"
        "addc.cc.u32 %7, %22, %22;\n\t"
        "addc.cc.u32 %8, %23, %23;\n\t"
        "addc.cc.u32 %9, %24, %24;\n\t"
        "addc.cc.u32 %10, %25, %25;\n\t"
        "addc.cc.u32 %11, %26, %26;\n\t"
        "addc.cc.u32 %12, %27, %27;\n\t"
        "addc.cc.u32 %13, %28, %28;\n\t"
        "addc.u32 %14, %29, %29;\n\t"
        : "=&r"(x1), "=&r"(x2), "=&r"(x3), "=&r"(x4), "=&r"(x5), "=&r"(x6), "=&r"(x7), "=&r"(x8), "=&r"(x9), "=&r"(x10), "=&r"(x11), "=&r"(x12), "=&r"(x13), "=&r"(x14), "=&r"(x15)
        : "r"(o0), "r"(s2), "r"(s3), "r"(s4), "r"(s5), "r"(s6), "r"(s7), "r"(s8), "r"(s9), "r"(s10), "r"(s11), "r"(s12), "r"(s13), "r"(s14), "r"(s15));
    // t = x + diagonal: (t0,t1) = a0^2, (t2,t3) = a1^2, ... one carry chain
    asm("mul.lo.u32 %0, %16, %16;\n\t"
        "mad.hi.cc.u32 %1, %16, %16, %24;\n\t"
        "madc.lo.cc.u32 %2, %17, %17, %25;\n\t madc.hi.cc.u32 %3, %17, %17, %26;\n\t"
        "madc.lo.cc.u32 %4, %18, %18, %27;\n\t madc.hi.cc.u32 %5, %18, %18, %28;\n\t"
        "madc.lo.cc.u32 %6, %19, %19, %29;\n\t madc.hi.cc.u32 %7, %19, %19, %30;\n\t"
        "madc.lo.cc.u32 %8, %20, %20, %31;\n\t madc.hi.cc.u32 %9, %20, %20, %32;\n\t"
        "madc.lo.cc.u32 %10, %21, %21, %33;\n\t madc.hi.cc.u32 %11, %21, %21, %34;\n\t"
        "madc.lo.cc.u32 %12, %22, %22, %35;\n\t madc.hi.cc.u32 %13, %22, %22, %36;\n\t"
        "madc.lo.cc.u32 %14, %23, %23, %37;\n\t madc.hi.u32 %15, %23, %23, %38;\n\t"
        : "=&r"(t[0]), "=&r"(t[1]), "=&r"(t[2]), "=&r"(t[3]), "=&r"(t[4]), "=&r"(t[5]), "=&r"(t[6]), "=&r"(t[7]),
          "=&r"(t[8]), "=&r"(t[9]), "=&r"(t[10]), "=&r"(t[11]), "=&r"(t[12]), "=&r"(t[13]), "=&r"(t[14]), "=&r"(t[15])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),
          "r"(x1), "r"(x2), "r"(x3), "r"(x4), "r"(x5), "r"(x6), "r"(x7), "r"(x8), "r"(x9), "r"(x10), "r"(x11), "r"(x12), "r"(x13), "r"(x14), "r"(x15));
#else
    fe_mul_wide(t, A, A);
#endif
}
BP_FEMUL fe fe_sq(const fe &a) { uint32_t t[16]; fe_sq_wide(t, a); return fe_reduce_wide(t); }
BP_HD fe fe_sqn(fe a, int n) {
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int i = 0; i < n; i++) a = fe_sq(a);
    return a;
}
BP_HD fe fe_dbl(const fe &a) { return fe_add(a, a); }

// canonical representative in [0, p)
BP_HD fe fe_canon(const fe &a) {
    fe r = a;
    // fold bit 255: v = (v mod 2^255) + 19*bit255  (< 2^255 + 19)
    uint64_t c = (uint64_t)(r.v[7] >> 31) * 19u;
    r.v[7] &= 0x7fffffffu;
    for (int i = 0; i < 8; i++) { c += r.v[i]; r.v[i] = (uint32_t)c; c >>= 32; }
    // v >= p  <=>  v + 19 >= 2^255
    fe s; c = 19;
    for (int i = 0; i < 8; i++) { c += r.v[i]; s.v[i] = (uint32_t)c; c >>= 32; }
    uint32_t ge_p = s.v[7] >> 31;            // 1 if v >= p; then v - p = (v + 19) - 2^255
    s.v[7] &= 0x7fffffffu;
    uint32_t m = 0u - ge_p;
    for (int i = 0; i < 8; i++) r.v[i] = (s.v[i] & m) | (r.v[i] & ~m);
    return r;
}
BP_HD void fe_tobytes(uint8_t out[32], const fe &a) {
    fe c = fe_canon(a);
    for (int i = 0; i < 8; i++) { out[4 * i] = (uint8_t)c.v[i]; out[4 * i + 1] = (uint8_t)(c.v[i] >> 8); out[4 * i + 2] = (uint8_t)(c.v[i] >> 16); out[4 * i + 3] = (uint8_t)(c.v[i] >> 24); }
}
// loads all 256 bits (callers decide what to do with bit 255 / non-canonical values)
BP_HD fe fe_frombytes_raw(const uint8_t in[32]) {
    fe r;
    for (int i = 0; i < 8; i++) r.v[i] = (uint32_t)in[4 * i] | ((uint32_t)in[4 * i + 1] << 8) | ((uint32_t)in[4 * i + 2] << 16) | ((uint32_t)in[4 * i + 3] << 24);
    return r;
}
BP_HD bool fe_is_negative(const fe &a) { return fe_canon(a).v[0] & 1u; }
BP_HD bool fe_is_zero(const fe &a) { fe c = fe_canon(a); uint32_t z = 0; for (int i = 0; i < 8; i++) z |= c.v[i]; return z == 0; }
BP_HD bool fe_eq(const fe &a, const fe &b) { return fe_is_zero(fe_sub(a, b)); }
BP_HD fe fe_select(const fe &a, const fe &b, bool pick_b) { fe r; uint32_t m = 0u - (uint32_t)pick_b; for (int i = 0; i < 8; i++) r.v[i] = (b.v[i] & m) | (a.v[i] & ~m); return r; }
BP_HD fe fe_cneg(const fe &a, bool neg) { return fe_select(a, fe_neg(a), neg); }
// mask-taking forms for secret conditions (msm_ct.cuh): mask is all-ones or zero and is never turned into a bool
BP_HD fe fe_select_mask(const fe &a, const fe &b, uint32_t mask) { fe r; for (int i = 0; i < 8; i++) r.v[i] = a.v[i] ^ ((a.v[i] ^ b.v[i]) & mask); return r; }
BP_HD fe fe_cneg_mask(const fe &a, uint32_t mask) { return fe_select_mask(a, fe_neg(a), mask); }
BP_HD fe fe_abs(const fe &a) { return fe_cneg(a, fe_is_negative(a)); }

// z^(2^250-1) with z^11 on the side: the shared ladder of invert and pow22523
BP_HDN fe fe_pow_2_250_1(const fe &z, fe &z11) {
    fe t0 = fe_sq(z);                          // 2
    fe t1 = fe_mul(z, fe_sqn(t0, 2));          // 9
    t0 = fe_mul(t0, t1);                       // 11
    z11 = t0;
    t1 = fe_mul(t1, fe_sq(t0));                // 2^5-1
    t1 = fe_mul(fe_sqn(t1, 5), t1);            // 2^10-1
    fe t2 = fe_mul(fe_sqn(t1, 10), t1);        // 2^20-1
    t2 = fe_mul(fe_sqn(t2, 20), t2);           // 2^40-1
    t1 = fe_mul(fe_sqn(t2, 10), t1);           // 2^50-1
    t2 = fe_mul(fe_sqn(t1, 50), t1);           // 2^100-1
    t2 = fe_mul(fe_sqn(t2, 100), t2);          // 2^200-1
    return fe_mul(fe_sqn(t2, 50), t1);         // 2^250-1
}
BP_HD fe fe_invert(const fe &z) { fe z11; fe t = fe_pow_2_250_1(z, z11); return fe_mul(fe_sqn(t, 5), z11); }
BP_HD fe fe_pow22523(const fe &z) { fe z11; fe t = fe_pow_2_250_1(z, z11); return fe_mul(fe_sqn(t, 2), z); }
