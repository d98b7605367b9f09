// TEST-ONLY compile-time audit of the constant-time MSM's secret-dependent code (bulletproofs_b200/csrc/msm_ct.cuh).
//
// The recoding and the selection are templates on their word type.  Here they are instantiated with Secret, a word that supports the
// arithmetic and bitwise operators the algorithms need but has no conversion to bool or to an integer and no comparison operators.
// A branch (if, ?:, &&, a loop condition), a comparison or an array index on a scalar-derived value therefore does not compile.
// tests/test_msm_ct_cpu.py builds this file with g++, and builds it once more with -DCT_AUDIT_NEGATIVE_CONTROL=<n>, which adds a
// snippet that does branch or index on a Secret: that build must fail, or the audit would prove nothing.
//
// What this does not cover: the field and group operations the selected point feeds (fe.cuh / ge.cuh are fixed carry chains on
// uint32_t, reviewed rather than type-checked) and the code the compiler emits (the SASS guard of the same test looks at that).
#include <cstdint>
#include "../../bulletproofs_b200/csrc/msm_ct.cuh"

struct Secret {
    uint32_t v_;                     // only the operators below may read it
    Secret() = default;
    Secret(uint32_t x) : v_(x) {}    // public -> secret is allowed; secret -> public is not
    explicit operator bool() const = delete;
};
#define CT_BIN(op)                                                                         \
    inline Secret operator op(Secret a, Secret b) { return Secret(a.v_ op b.v_); }         \
    inline Secret operator op(Secret a, uint32_t b) { return Secret(a.v_ op b); }          \
    inline Secret operator op(uint32_t a, Secret b) { return Secret(a op b.v_); }
CT_BIN(+) CT_BIN(-) CT_BIN(*) CT_BIN(&) CT_BIN(|) CT_BIN(^)
#undef CT_BIN
inline Secret operator~(Secret a) { return Secret(~a.v_); }
inline Secret operator<<(Secret a, int s) { return Secret(a.v_ << s); }         // shift counts are public
inline Secret operator>>(Secret a, int s) { return Secret(a.v_ >> s); }

// every template of msm_ct.cuh that touches a scalar, instantiated on Secret words
void audit(const Secret scalar[8], const uint32_t *table, Secret out[32], Secret digits[CT_DIGITS]) {
    Secret s[8];
    Secret bad = ct_scalar_geq_l_mask(scalar);
    for (int i = 0; i < 8; i++) s[i] = scalar[i] & ~bad;
    ct_recode_radix16(s, digits);
    for (int w = 0; w < CT_DIGITS; w++) {
        Secret neg, abs;
        ct_digit_split(digits[w], neg, abs);
        ct_select_entry(abs, [&](uint32_t j, int k, uint32_t *q) { for (int i = 0; i < 4; i++) q[i] = table[32 * j + k + i]; }, out);
        for (int k = 0; k < 32; k++) out[k] = out[k] ^ (neg & 0u);
    }
    (void)ct_mask_eq(s[0], 7u);
}

#if defined(CT_AUDIT_NEGATIVE_CONTROL)
// each of these must be rejected by the compiler
uint32_t negative_control(Secret d, const uint32_t *table) {
#if CT_AUDIT_NEGATIVE_CONTROL == 1
    if (d) return table[0];                          // branch on a secret
    return 0;
#elif CT_AUDIT_NEGATIVE_CONTROL == 2
    return table[d];                                 // index with a secret
#else
    return d == Secret(3u) ? table[1] : table[2];    // compare a secret
#endif
}
#endif
