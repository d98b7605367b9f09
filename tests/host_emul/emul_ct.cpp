// TEST-ONLY host build of the constant-time indexed MSM (bulletproofs_b200/csrc/msm_ct.cuh) with g++: the same recoding, canonicality
// mask, [1..8]P tables, masked lookups and chunked Straus loop as the k_msm_ct_* kernels, so that the CPU tier can check them against
// the oracle without a GPU.  tests/test_msm_ct_cpu.py compiles this file into a temporary directory.  Nothing in the product links it.
#include <algorithm>
#include <cstring>
#include <vector>
#include "../../bulletproofs_b200/csrc/ge.cuh"
#include "../../bulletproofs_b200/csrc/sc.cuh"
#include "../../bulletproofs_b200/csrc/msm_ct.cuh"

extern "C" {

// points: T compressed points (one per term); outs: n_msm x 32 B; status[j] = 3 (BP_ERR_NONCANONICAL_SCALAR) or 0.  Chunks of at most
// `ch` terms, cut at MSM boundaries; per MSM the chunk partials are added up.  Returns 1 for an undecodable point.
int emul_msm_ct(const uint8_t *scalars, const uint8_t *points, const uint64_t *offsets, uint32_t n_msm, uint32_t ch, uint8_t *outs, uint8_t *status) {
    const uint32_t T = (uint32_t)offsets[n_msm];
    std::vector<ge_ext> tab((size_t)T * CT_TABLE);
    std::vector<int8_t> digits((size_t)T * CT_DIGITS);
    std::vector<uint32_t> bad(n_msm, 0);
    for (uint32_t j = 0; j < n_msm; j++)
        for (uint32_t t = (uint32_t)offsets[j]; t < offsets[j + 1]; t++) {
            fe x, y; if (!ge_decode(x, y, points + 32 * (size_t)t)) return 1;
            ct_table(ge_from_niels(ge_to_niels_affine(x, y)), [&](int k, const ge_ext &p) { tab[(size_t)CT_TABLE * t + k] = p; });
            uint32_t s[8]; sc l = sc_load(scalars + 32 * (size_t)t); for (int i = 0; i < 8; i++) s[i] = l.v[i];
            uint32_t m = ct_scalar_geq_l_mask(s);
            for (int i = 0; i < 8; i++) s[i] &= ~m;
            uint32_t d[CT_DIGITS]; ct_recode_radix16(s, d);
            for (int i = 0; i < CT_DIGITS; i++) digits[(size_t)CT_DIGITS * t + i] = (int8_t)(uint8_t)d[i];
            bad[j] |= m & 1u;
        }
    for (uint32_t j = 0; j < n_msm; j++) {
        ge_ext sum = ge_identity();
        for (uint32_t lo = (uint32_t)offsets[j]; lo < offsets[j + 1]; lo += ch) {
            uint32_t hi = std::min<uint32_t>(lo + ch, (uint32_t)offsets[j + 1]);
            ge_ext acc = ge_identity();
            for (int w = CT_DIGITS - 1; w >= 0; w--) {
                if (w != CT_DIGITS - 1) for (int i = 0; i < 4; i++) acc = ge_dbl(acc);
                for (uint32_t t = lo; t < hi; t++) {
                    const uint32_t *base = reinterpret_cast<const uint32_t *>(&tab[(size_t)CT_TABLE * t]);
                    acc = ge_add(acc, ct_lookup((uint32_t)(int32_t)digits[(size_t)CT_DIGITS * t + w], [&](uint32_t e, int k, uint32_t *v) { memcpy(v, base + 32 * e + k, 16); }));
                }
            }
            sum = ge_add(sum, acc);
        }
        ge_encode(outs + 32 * j, sum);
        status[j] = bad[j] ? 3 : 0;
    }
    return 0;
}
// signed radix-16 recoding of one 32-byte scalar (the canonicality mask is not applied): 64 digits as signed bytes
void emul_ct_recode(const uint8_t *scalar, int8_t *digits) {
    uint32_t s[8]; sc l = sc_load(scalar); for (int i = 0; i < 8; i++) s[i] = l.v[i];
    uint32_t d[CT_DIGITS]; ct_recode_radix16(s, d);
    for (int i = 0; i < CT_DIGITS; i++) digits[i] = (int8_t)(uint8_t)d[i];
}
int emul_ct_geq_l(const uint8_t *scalar) { uint32_t s[8]; sc l = sc_load(scalar); for (int i = 0; i < 8; i++) s[i] = l.v[i]; return (int)(ct_scalar_geq_l_mask(s) & 1u); }
}
