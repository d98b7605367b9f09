// Host mirror of the reference protocol layer (see bulletproofs.hpp).  Point arithmetic: libbpmsm.so only.
#include "bulletproofs.hpp"

namespace bulletproofs {

// ------------------------------------------------------------------ ChaChaRng
static inline uint32_t rotl32(uint32_t x, int n) { return (x << n) | (x >> (32 - n)); }
void ChaChaRng::block() {
    uint32_t in[16] = {0x61707865, 0x3320646e, 0x79622d32, 0x6b206574}, x[16];
    memcpy(in + 4, key_, 32);
    in[12] = (uint32_t)counter_; in[13] = (uint32_t)(counter_ >> 32); in[14] = 0; in[15] = 0;
    memcpy(x, in, 64);
    auto qr = [&](int a, int b, int c, int d) {
        x[a] += x[b]; x[d] = rotl32(x[d] ^ x[a], 16); x[c] += x[d]; x[b] = rotl32(x[b] ^ x[c], 12);
        x[a] += x[b]; x[d] = rotl32(x[d] ^ x[a], 8);  x[c] += x[d]; x[b] = rotl32(x[b] ^ x[c], 7);
    };
    for (int i = 0; i < 10; i++) { qr(0, 4, 8, 12); qr(1, 5, 9, 13); qr(2, 6, 10, 14); qr(3, 7, 11, 15); qr(0, 5, 10, 15); qr(1, 6, 11, 12); qr(2, 7, 8, 13); qr(3, 4, 9, 14); }
    for (int i = 0; i < 16; i++) x[i] += in[i];
    memcpy(buf_, x, 64); counter_++; used_ = 0;
}
void ChaChaRng::fill_bytes(uint8_t *out, size_t n) { for (size_t i = 0; i < n; i++) { if (used_ == 64) block(); out[i] = buf_[used_++]; } }

Scalar inner_product(const std::vector<Scalar> &a, const std::vector<Scalar> &b) {       // inner_product_proof.rs:418-427
    if (a.size() != b.size()) throw std::invalid_argument("inner_product: lengths differ");
    const size_t n = a.size(), chunk = 4096;
    if (n <= chunk) { Scalar acc = Scalar::zero(); for (size_t i = 0; i < n; i++) acc += a[i] * b[i]; return acc; }
    std::vector<Scalar> part((n + chunk - 1) / chunk, Scalar::zero());        // long vectors (R1CS): partial sums over the host cores
    parallel_for(part.size(), [&](size_t c) { Scalar acc = Scalar::zero(); for (size_t i = c * chunk; i < std::min(n, (c + 1) * chunk); i++) acc += a[i] * b[i]; part[c] = acc; });
    Scalar acc = Scalar::zero(); for (const Scalar &x : part) acc += x;
    return acc;
}


static void check(int rc, bp_ctx *ctx, const char *what) {
    if (rc == BP_OK) return;
    throw std::runtime_error(std::string(what) + " failed with code " + std::to_string(rc) + ": " + bp_last_error(ctx));
}
static std::vector<uint8_t> pack(const std::vector<Scalar> &v) { std::vector<uint8_t> o(32 * v.size()); for (size_t i = 0; i < v.size(); i++) v[i].write(o.data() + 32 * i); return o; }

// ------------------------------------------------------------------ InnerProductProof::create
// The round loop of inner_product_proof.rs:69-185 against a device session that holds a, b, the factor / challenge coefficient vectors and
// the (never folded) generators of B proofs of the same length: per round one bp_ippx_round (L, R of every proof), the transcripts on the
// host, one bp_ippx_fold.  ts[p] is proof p's transcript.
static std::vector<InnerProductProof> ipp_rounds_x(bp_ippx *sess, bp_ctx *ctx, std::vector<Transcript *> &ts, size_t n) {
    size_t B = ts.size();
    for (Transcript *t : ts) t->innerproduct_domain_sep(n);
    std::vector<InnerProductProof> proofs(B);
    std::vector<uint8_t> lr(64 * B), u(32 * B), ui(32 * B), ab(64 * B);
    while (n != 1) {
        check(bp_ippx_round(sess, lr.data()), ctx, "bp_ippx_round");
        parallel_for(B, [&](size_t p) {
            CompressedRistretto L, R; memcpy(L.data(), lr.data() + 64 * p, 32); memcpy(R.data(), lr.data() + 64 * p + 32, 32);
            proofs[p].L_vec.push_back(L); proofs[p].R_vec.push_back(R);
            ts[p]->append_point("L", L); ts[p]->append_point("R", R);
            Scalar c = ts[p]->challenge_scalar("u"), ci = c.invert();
            Bytes32 cb = c.to_bytes(), cib = ci.to_bytes(); memcpy(u.data() + 32 * p, cb.data(), 32); memcpy(ui.data() + 32 * p, cib.data(), 32);
        });
        check(bp_ippx_fold(sess, u.data(), ui.data()), ctx, "bp_ippx_fold");
        n /= 2;
    }
    check(bp_ippx_finish(sess, ab.data()), ctx, "bp_ippx_finish");
    for (size_t p = 0; p < B; p++)
        if (!Scalar::from_canonical_bytes(ab.data() + 64 * p, proofs[p].a) || !Scalar::from_canonical_bytes(ab.data() + 64 * p + 32, proofs[p].b)) throw std::runtime_error("bp_ippx_finish: bad scalar");
    return proofs;
}
static void ipp_check_lengths(size_t n, const std::vector<Scalar> &Gf, const std::vector<Scalar> &Hf, const std::vector<Scalar> &a, const std::vector<Scalar> &b) {
    if (b.size() != n || Gf.size() != n || Hf.size() != n || a.size() != n) throw std::invalid_argument("InnerProductProof::create: vector lengths differ");   // :59-64
    if (n == 0 || (n & (n - 1))) throw std::invalid_argument("InnerProductProof::create: length must be a power of two");                              // :67
}

InnerProductProof InnerProductProof::create(Device &dev, const BulletproofGens &gens, size_t n, size_t m, Transcript &t, const CompressedRistretto &Q,
                                            const std::vector<Scalar> &Gf, const std::vector<Scalar> &Hf, std::vector<Scalar> a, std::vector<Scalar> b) {
    ipp_check_lengths(n * m, Gf, Hf, a, b);
    bp_ippx *sess = nullptr;
    check(bp_ippx_begin(dev.ctx, gens.handle, n, m, 1, Q.data(), pack(Gf).data(), pack(Hf).data(), pack(a).data(), pack(b).data(), &sess), dev.ctx, "bp_ippx_begin");
    std::vector<Transcript *> ts = {&t};
    try { InnerProductProof p = ipp_rounds_x(sess, dev.ctx, ts, n * m)[0]; bp_ippx_end(sess); return p; }
    catch (...) { bp_ippx_end(sess); throw; }
}
InnerProductProof InnerProductProof::create(Device &dev, Transcript &t, const CompressedRistretto &Q, const std::vector<Scalar> &Gf, const std::vector<Scalar> &Hf,
                                            const std::vector<CompressedRistretto> &G, const std::vector<CompressedRistretto> &H, std::vector<Scalar> a, std::vector<Scalar> b) {
    if (G.size() != a.size() || H.size() != a.size()) throw std::invalid_argument("InnerProductProof::create: vector lengths differ");
    ipp_check_lengths(a.size(), Gf, Hf, a, b);
    bp_ippx *sess = nullptr;
    check(bp_ippx_begin_points(dev.ctx, G[0].data(), H[0].data(), G.size(), 1, Q.data(), pack(Gf).data(), pack(Hf).data(), pack(a).data(), pack(b).data(), &sess), dev.ctx, "bp_ippx_begin_points");
    std::vector<Transcript *> ts = {&t};
    try { InnerProductProof p = ipp_rounds_x(sess, dev.ctx, ts, a.size())[0]; bp_ippx_end(sess); return p; }
    catch (...) { bp_ippx_end(sess); throw; }
}
// B proofs over the same generators G(n, m), H(n, m) in one device session (every MSM launch chain carries all proofs)
std::vector<InnerProductProof> InnerProductProof::create_many(Device &dev, const BulletproofGens &gens, size_t n, size_t m, std::vector<Transcript *> &ts, const std::vector<CompressedRistretto> &Qs,
                                                              const std::vector<std::vector<Scalar>> &Gfs, const std::vector<std::vector<Scalar>> &Hfs,
                                                              const std::vector<std::vector<Scalar>> &as, const std::vector<std::vector<Scalar>> &bs) {
    size_t B = ts.size(), N = n * m;
    if (Qs.size() != B || Gfs.size() != B || Hfs.size() != B || as.size() != B || bs.size() != B || B == 0) throw std::invalid_argument("InnerProductProof::create_many: batch sizes differ");
    std::vector<uint8_t> q(32 * B), gf(32 * B * N), hf(32 * B * N), av(32 * B * N), bv(32 * B * N);
    parallel_for(B, [&](size_t p) {
        ipp_check_lengths(N, Gfs[p], Hfs[p], as[p], bs[p]);
        memcpy(q.data() + 32 * p, Qs[p].data(), 32);
        memcpy(gf.data() + 32 * N * p, pack(Gfs[p]).data(), 32 * N); memcpy(hf.data() + 32 * N * p, pack(Hfs[p]).data(), 32 * N);
        memcpy(av.data() + 32 * N * p, pack(as[p]).data(), 32 * N); memcpy(bv.data() + 32 * N * p, pack(bs[p]).data(), 32 * N);
    });
    bp_ippx *sess = nullptr;
    check(bp_ippx_begin(dev.ctx, gens.handle, n, m, B, q.data(), gf.data(), hf.data(), av.data(), bv.data(), &sess), dev.ctx, "bp_ippx_begin");
    try { std::vector<InnerProductProof> out = ipp_rounds_x(sess, dev.ctx, ts, N); bp_ippx_end(sess); return out; }
    catch (...) { bp_ippx_end(sess); throw; }
}

ProofError InnerProductProof::verification_scalars(size_t n, Transcript &t, std::vector<Scalar> &u_sq, std::vector<Scalar> &u_inv_sq, std::vector<Scalar> &s) const {
    size_t lg_n = L_vec.size();
    if (lg_n >= 32) return ProofError::VerificationError;
    if (n != ((size_t)1 << lg_n)) return ProofError::VerificationError;
    t.innerproduct_domain_sep(n);
    std::vector<Scalar> ch(lg_n), chi(lg_n);
    for (size_t i = 0; i < lg_n; i++) {
        if (!t.validate_and_append_point("L", L_vec[i]) || !t.validate_and_append_point("R", R_vec[i])) return ProofError::VerificationError;
        ch[i] = t.challenge_scalar("u");
    }
    // Scalar::batch_invert: every inverse and the product of all inverses (:226-227), one field inversion
    std::vector<Scalar> pre(lg_n + 1); pre[0] = Scalar::one();
    for (size_t i = 0; i < lg_n; i++) pre[i + 1] = pre[i] * ch[i];
    Scalar inv = pre[lg_n].invert(), allinv = inv;
    for (size_t i = lg_n; i-- > 0;) { chi[i] = inv * pre[i]; inv = inv * ch[i]; }
    u_sq.resize(lg_n); u_inv_sq.resize(lg_n);
    for (size_t i = 0; i < lg_n; i++) { u_sq[i] = ch[i] * ch[i]; u_inv_sq[i] = chi[i] * chi[i]; }
    s.resize(n); s[0] = allinv;
    for (size_t i = 1; i < n; i++) {
        size_t lg_i = 63 - (size_t)__builtin_clzll((unsigned long long)i), k = (size_t)1 << lg_i;
        s[i] = s[i - k] * u_sq[(lg_n - 1) - lg_i];
    }
    return ProofError::Ok;
}

ProofError InnerProductProof::verify(Device &dev, size_t n, Transcript &t, const std::vector<Scalar> &Gf, const std::vector<Scalar> &Hf, const CompressedRistretto &P,
                                     const CompressedRistretto &Q, const std::vector<CompressedRistretto> &G, const std::vector<CompressedRistretto> &H) const {
    std::vector<Scalar> u_sq, u_inv_sq, s;
    ProofError e = verification_scalars(n, t, u_sq, u_inv_sq, s);
    if (e != ProofError::Ok) return e;
    size_t k = L_vec.size(), nt = 1 + 2 * n + 2 * k;
    std::vector<Scalar> sc_(nt); std::vector<uint8_t> pts(32 * nt);
    sc_[0] = a * b; memcpy(pts.data(), Q.data(), 32);
    for (size_t i = 0; i < n; i++) {
        sc_[1 + i] = (a * s[i]) * Gf[i]; memcpy(pts.data() + 32 * (1 + i), G[i].data(), 32);
        sc_[1 + n + i] = (b * s[n - 1 - i]) * Hf[i]; memcpy(pts.data() + 32 * (1 + n + i), H[i].data(), 32);
    }
    for (size_t i = 0; i < k; i++) {
        sc_[1 + 2 * n + i] = -u_sq[i]; memcpy(pts.data() + 32 * (1 + 2 * n + i), L_vec[i].data(), 32);
        sc_[1 + 2 * n + k + i] = -u_inv_sq[i]; memcpy(pts.data() + 32 * (1 + 2 * n + k + i), R_vec[i].data(), 32);
    }
    CompressedRistretto expect;
    int rc = bp_msm(dev.ctx, pack(sc_).data(), pts.data(), nt, expect.data());
    if (rc == BP_ERR_INVALID_POINT) return ProofError::VerificationError;       // decompress() -> None (:296-306)
    check(rc, dev.ctx, "bp_msm");
    return expect == P ? ProofError::Ok : ProofError::VerificationError;         // canonical encodings: equal bytes <=> equal points (:321)
}

std::vector<uint8_t> InnerProductProof::to_bytes() const {
    std::vector<uint8_t> buf;
    for (size_t i = 0; i < L_vec.size(); i++) { buf.insert(buf.end(), L_vec[i].begin(), L_vec[i].end()); buf.insert(buf.end(), R_vec[i].begin(), R_vec[i].end()); }
    Bytes32 ab = a.to_bytes(); buf.insert(buf.end(), ab.begin(), ab.end());
    ab = b.to_bytes(); buf.insert(buf.end(), ab.begin(), ab.end());
    return buf;
}
ProofError InnerProductProof::from_bytes(const uint8_t *s, size_t len, InnerProductProof &out) {
    if (len % 32 != 0) return ProofError::FormatError;
    size_t ne = len / 32;
    if (ne < 2 || (ne - 2) % 2 != 0) return ProofError::FormatError;
    size_t lg_n = (ne - 2) / 2;
    if (lg_n >= 32) return ProofError::FormatError;
    out.L_vec.resize(lg_n); out.R_vec.resize(lg_n);
    for (size_t i = 0; i < lg_n; i++) { memcpy(out.L_vec[i].data(), s + 64 * i, 32); memcpy(out.R_vec[i].data(), s + 64 * i + 32, 32); }
    if (!Scalar::from_canonical_bytes(s + 64 * lg_n, out.a) || !Scalar::from_canonical_bytes(s + 64 * lg_n + 32, out.b)) return ProofError::FormatError;
    return ProofError::Ok;
}

// ------------------------------------------------------------------ LinearProof
// The device session of the inner-product prover is reused: G stays on the device and is folded there; the session's
// H vector is filled with copies of B and its Q slot holds F, so that one bp_ipp_lr call gives
//   L = <a_L, G_R> + s_j B + c_L F   and   R = <a_R, G_L> + t_j B + c_R F        (linear_proof.rs:96-107).
static void linear_transcript_header(Transcript &t, size_t n, const CompressedRistretto &C, const std::vector<Scalar> &b, const std::vector<CompressedRistretto> &G,
                                     const CompressedRistretto &F, const CompressedRistretto &B) {
    t.innerproduct_domain_sep(n);
    t.append_point("C", C);
    for (const Scalar &bi : b) t.append_scalar("b_i", bi);
    for (const CompressedRistretto &g : G) t.append_point("G_i", g);
    t.append_point("F", F); t.append_point("B", B);
}
ProofError LinearProof::create(Device &dev, Transcript &t, Rng &rng, const CompressedRistretto &C, Scalar r, std::vector<Scalar> a, std::vector<Scalar> b,
                               const std::vector<CompressedRistretto> &G, const CompressedRistretto &F, const CompressedRistretto &B, LinearProof &out) {
    size_t n = b.size(), n0 = n;
    if (G.size() != n) return ProofError::InvalidGeneratorsLength;
    if (a.size() != n || n == 0 || (n & (n - 1))) return ProofError::InvalidInputLength;
    linear_transcript_header(t, n, C, b, G, F, B);
    out.L_vec.clear(); out.R_vec.clear();
    bp_ipp *sess = nullptr;
    if (n0 >= 2) {
        std::vector<CompressedRistretto> H(n0, B);
        check(bp_ipp_begin_points(dev.ctx, G[0].data(), H[0].data(), n0, F.data(), &sess), dev.ctx, "bp_ipp_begin_points");
    }
    try {
        Scalar one = Scalar::one(), zero = Scalar::zero();
        while (n != 1) {
            n /= 2;
            std::vector<Scalar> aL(a.begin(), a.begin() + n), aR(a.begin() + n, a.begin() + 2 * n), bL(b.begin(), b.begin() + n), bR(b.begin() + n, b.begin() + 2 * n);
            Scalar c_L = inner_product(aL, bR), c_R = inner_product(aR, bL);
            Scalar s_j = Scalar::random(rng), t_j = Scalar::random(rng);
            std::vector<Scalar> sL(2 * n + 1, zero), sR(2 * n + 1, zero);
            for (size_t i = 0; i < n; i++) { sL[i] = aL[i]; sR[i] = aR[i]; }
            sL[n] = s_j; sR[n] = t_j; sL[2 * n] = c_L; sR[2 * n] = c_R;
            CompressedRistretto L, R;
            check(bp_ipp_lr(sess, n, pack(sL).data(), pack(sR).data(), L.data(), R.data()), dev.ctx, "bp_ipp_lr");
            out.L_vec.push_back(L); out.R_vec.push_back(R);
            t.append_point("L", L); t.append_point("R", R);
            Scalar x = t.challenge_scalar("x_j"), x_inv = x.invert();
            for (size_t i = 0; i < n; i++) { a[i] = aL[i] + x_inv * aR[i]; b[i] = bL[i] + x * bR[i]; }      // :124-126
            check(bp_ipp_fold(sess, n, one.to_bytes().data(), x.to_bytes().data(), one.to_bytes().data(), zero.to_bytes().data(), 0), dev.ctx, "bp_ipp_fold");   // G_L += x G_R (:127-131)
            a.resize(n); b.resize(n);
            r = r + x * s_j + x_inv * t_j;
        }
        Scalar s_star = Scalar::random(rng), t_star = Scalar::random(rng);
        // S = t* B + s* b_0 F + s* G_0   (:143)
        if (n0 >= 2) {
            std::vector<Scalar> sL(3, zero), sR = {s_star, t_star, s_star * b[0]};
            CompressedRistretto junk;
            check(bp_ipp_lr(sess, 1, pack(sL).data(), pack(sR).data(), junk.data(), out.S.data()), dev.ctx, "bp_ipp_lr");
        } else {
            std::vector<Scalar> s3 = {t_star, s_star * b[0], s_star}; uint8_t pts[96];
            memcpy(pts, B.data(), 32); memcpy(pts + 32, F.data(), 32); memcpy(pts + 64, G[0].data(), 32);
            check(bp_msm(dev.ctx, pack(s3).data(), pts, 3, out.S.data()), dev.ctx, "bp_msm");
        }
        t.append_point("S", out.S);
        Scalar x_star = t.challenge_scalar("x_star");
        out.a = s_star + x_star * a[0]; out.r = t_star + x_star * r;
        if (sess) bp_ipp_end(sess);
        return ProofError::Ok;
    } catch (...) { if (sess) bp_ipp_end(sess); throw; }
}
ProofError LinearProof::verify(Device &dev, Transcript &t, const CompressedRistretto &C, const std::vector<CompressedRistretto> &G, const CompressedRistretto &F,
                               const CompressedRistretto &B, std::vector<Scalar> b) const {
    size_t n = b.size(), lg_n = L_vec.size();
    if (G.size() != n) return ProofError::InvalidGeneratorsLength;
    linear_transcript_header(t, n, C, b, G, F, B);
    if (lg_n >= 32 || n != ((size_t)1 << lg_n)) return ProofError::VerificationError;           // verification_scalars :235-241
    std::vector<Scalar> x(lg_n), x_inv(lg_n);
    size_t nm = n;
    for (size_t j = 0; j < lg_n; j++) {
        if (!t.validate_and_append_point("L", L_vec[j]) || !t.validate_and_append_point("R", R_vec[j])) return ProofError::VerificationError;
        x[j] = t.challenge_scalar("x_j");
        nm /= 2;
        for (size_t i = 0; i < nm; i++) b[i] = b[i] + x[j] * b[nm + i];
    }
    for (size_t j = 0; j < lg_n; j++) x_inv[j] = x[j].invert();
    t.append_point("S", S);
    Scalar x_star = t.challenge_scalar("x_star");
    // expect_S = r B + a b_0 F - x*(C + sum x_j L_j + sum x_j^-1 R_j) + a sum s_i G_i   (:208-218) as one MSM
    std::vector<Scalar> sc_; std::vector<uint8_t> pts;
    auto term = [&](const Scalar &s_, const CompressedRistretto &p) { sc_.push_back(s_); pts.insert(pts.end(), p.begin(), p.end()); };
    term(r, B); term(a * b[0], F); term(-x_star, C);
    for (size_t j = 0; j < lg_n; j++) term(-(x_star * x[j]), L_vec[j]);
    for (size_t j = 0; j < lg_n; j++) term(-(x_star * x_inv[j]), R_vec[j]);
    std::vector<Scalar> s(n); s[0] = Scalar::one();
    for (size_t i = 1; i < n; i++) { size_t lg_i = 63 - (size_t)__builtin_clzll((unsigned long long)i); s[i] = s[i - ((size_t)1 << lg_i)] * x[(lg_n - 1) - lg_i]; }   // subset_product :272-284
    for (size_t i = 0; i < n; i++) term(a * s[i], G[i]);
    CompressedRistretto expect;
    int rc = bp_msm(dev.ctx, pack(sc_).data(), pts.data(), sc_.size(), expect.data());
    if (rc == BP_ERR_INVALID_POINT) return ProofError::VerificationError;
    check(rc, dev.ctx, "bp_msm");
    uint8_t ok = 0; check(bp_decompress_check_batch(dev.ctx, S.data(), 1, &ok), dev.ctx, "decompress S");       // S.decompress() must succeed (:204)
    return (ok && expect == S) ? ProofError::Ok : ProofError::VerificationError;
}
std::vector<uint8_t> LinearProof::to_bytes() const {
    std::vector<uint8_t> buf;
    for (size_t i = 0; i < L_vec.size(); i++) { buf.insert(buf.end(), L_vec[i].begin(), L_vec[i].end()); buf.insert(buf.end(), R_vec[i].begin(), R_vec[i].end()); }
    buf.insert(buf.end(), S.begin(), S.end());
    Bytes32 x = a.to_bytes(); buf.insert(buf.end(), x.begin(), x.end());
    x = r.to_bytes(); buf.insert(buf.end(), x.begin(), x.end());
    return buf;
}
ProofError LinearProof::from_bytes(const uint8_t *s, size_t len, LinearProof &out) {
    if (len % 32 != 0) return ProofError::FormatError;
    size_t ne = len / 32;
    if (ne < 3 || (ne - 3) % 2 != 0) return ProofError::FormatError;
    size_t lg_n = (ne - 3) / 2;
    if (lg_n >= 32) return ProofError::FormatError;
    out.L_vec.resize(lg_n); out.R_vec.resize(lg_n);
    for (size_t i = 0; i < lg_n; i++) { memcpy(out.L_vec[i].data(), s + 64 * i, 32); memcpy(out.R_vec[i].data(), s + 64 * i + 32, 32); }
    memcpy(out.S.data(), s + 64 * lg_n, 32);
    if (!Scalar::from_canonical_bytes(s + 64 * lg_n + 32, out.a) || !Scalar::from_canonical_bytes(s + 64 * lg_n + 64, out.r)) return ProofError::FormatError;
    return ProofError::Ok;
}

// ------------------------------------------------------------------ RangeProof
Scalar scalar_exp_vartime(const Scalar &x, uint64_t n) {      // util.rs:222-234
    Scalar result = Scalar::one(), aux = x;
    while (n > 0) { if (n & 1) result = result * aux; n >>= 1; aux = aux * aux; }
    return result;
}

// Per-proof prover state between the batched device calls of prove_many
namespace {
struct ProverState {
    size_t m = 0, N = 0; bool live = false;
    std::vector<Scalar> a_bl, s_bl, sL, sR, l0, l1, r0, r1, t0, t1, t2, t1_bl, t2_bl, offset_zz, l_vec, r_vec, Gf, Hf;
    Scalar y, z, zz, x, w;
    CompressedRistretto Q;
    size_t out_base = 0;        // first output slot of this proof in the current batched call
};
// the MSMs one proof asks for in a phase (scalars, table slots, end offsets), built per proof in parallel and merged into one device call
struct MsmReq { std::vector<Scalar> sc; std::vector<uint32_t> idx; std::vector<uint64_t> off; };
// the two indexed-MSM entry points with one signature: constant-time for secret scalars (phases 1-2), variable-time for Q = w B (phase 3)
using IndexedMsm = int (*)(bp_ctx *, bp_gens *, const uint8_t *, const uint32_t *, const uint64_t *, size_t, uint8_t *, uint8_t *);
int indexed_msm_vartime(bp_ctx *c, bp_gens *g, const uint8_t *sc, const uint32_t *idx, const uint64_t *off, size_t n_msm, uint8_t *out, uint8_t *st) {
    return bp_msm_indexed_batch(c, g, sc, idx, nullptr, 0, off, n_msm, out, st);
}
bool run_requests(Device &dev, const BulletproofGens &gens, IndexedMsm msm, const std::vector<MsmReq> &reqs, std::vector<ProverState> &st, std::vector<uint8_t> &out) {
    size_t terms = 0, n_msm = 0;
    for (const MsmReq &r : reqs) { terms += r.sc.size(); n_msm += r.off.size(); }
    if (n_msm == 0) return false;
    std::vector<uint8_t> sc(32 * terms); std::vector<uint32_t> idx(terms); std::vector<uint64_t> off(n_msm + 1); std::vector<size_t> base(reqs.size());
    size_t t0 = 0, m0 = 0; off[0] = 0;
    for (size_t p = 0; p < reqs.size(); p++) { base[p] = t0; st[p].out_base = m0; for (uint64_t e : reqs[p].off) off[++m0] = t0 + e; t0 += reqs[p].sc.size(); }
    parallel_for(reqs.size(), [&](size_t p) {
        for (size_t i = 0; i < reqs[p].sc.size(); i++) { reqs[p].sc[i].write(sc.data() + 32 * (base[p] + i)); idx[base[p] + i] = reqs[p].idx[i]; }
    });
    out.assign(32 * n_msm, 0); std::vector<uint8_t> stt(n_msm);
    check(msm(dev.ctx, gens.handle, sc.data(), idx.data(), off.data(), n_msm, out.data(), stt.data()), dev.ctx, "indexed MSM");
    return true;
}
}  // namespace

// RangeProof::prove_multiple_with_rng (range_proof/mod.rs:234-288; the MPC run with itself, party.rs / dealer.rs) for a batch of proofs.
// Each proof follows exactly the statement order of the single-proof flow (same transcript, same RNG draw order, App. A.2 of SURVEY.md);
// only the device calls are shared: phase 1 = all V_j, A, S; phase 2 = all T_1, T_2; phase 3 = all Q = w B; phase 4 = all inner-product proofs.
void RangeProof::prove_many(Device &dev, const BulletproofGens &gens, size_t n, std::vector<RangeProofJob> &jobs) {
    const size_t B = jobs.size();
    std::vector<ProverState> st(B);
    const Scalar one = Scalar::one();
    // ---- phase 1: parameter checks, RNG draws, bit commitments
    {
        std::vector<MsmReq> reqs(B);
        parallel_for(B, [&](size_t p) {
            RangeProofJob &J = jobs[p]; ProverState &S = st[p];
            std::vector<Scalar> &sc = reqs[p].sc; std::vector<uint32_t> &idx = reqs[p].idx; std::vector<uint64_t> &off = reqs[p].off;
            size_t m = J.values.size();
            if (m != J.blindings.size()) { J.error = ProofError::WrongNumBlindingFactors; return; }                   // mod.rs:246-248
            if (!(n == 8 || n == 16 || n == 32 || n == 64)) { J.error = ProofError::InvalidBitsize; return; }       // dealer.rs:44-46
            if (m == 0 || (m & (m - 1))) { J.error = ProofError::InvalidAggregation; return; }                      // dealer.rs:47-49
            if (gens.gens_capacity < n || gens.party_capacity < m) { J.error = ProofError::InvalidGeneratorsLength; return; }   // dealer.rs:50-55
            S.m = m; S.N = n * m; S.live = true;
            J.t->rangeproof_domain_sep(n, m);                                                                          // dealer.rs:70
            // RNG order per party: a_blinding, s_blinding, s_L[0..n), s_R[0..n)  (party.rs:98,114-116)
            S.a_bl.resize(m); S.s_bl.resize(m); S.sL.resize(S.N); S.sR.resize(S.N);
            for (size_t j = 0; j < m; j++) {
                S.a_bl[j] = Scalar::random(*J.rng); S.s_bl[j] = Scalar::random(*J.rng);
                for (size_t i = 0; i < n; i++) S.sL[j * n + i] = Scalar::random(*J.rng);
                for (size_t i = 0; i < n; i++) S.sR[j * n + i] = Scalar::random(*J.rng);
            }
            // m + 2 constant-base MSMs: V_j = v_j B + v~_j B~ (party.rs:51), A = sum_j (a~_j B~ + sum_i [bit ? G : -H]) (party.rs:100-112,
            // dealer.rs:112-113), S = sum_j (s~_j B~ + <s_L, G_j> + <s_R, H_j>) (party.rs:119-124, dealer.rs:115-116).  A is written with
            // every G_i and H_i present, sum_i (b_i G_i + (b_i - 1) H_i): the same point, with point indices that do not depend on the bits.
            for (size_t j = 0; j < m; j++) { sc.push_back(Scalar::from_u64(J.values[j])); idx.push_back(gens.slot_B()); sc.push_back(J.blindings[j]); idx.push_back(gens.slot_B_blinding()); off.push_back(sc.size()); }
            for (size_t j = 0; j < m; j++) {
                sc.push_back(S.a_bl[j]); idx.push_back(gens.slot_B_blinding());
                for (size_t i = 0; i < n; i++) { Scalar b = Scalar::from_u64((J.values[j] >> i) & 1); sc.push_back(b); idx.push_back(gens.slot_G(j, i)); sc.push_back(b - one); idx.push_back(gens.slot_H(j, i)); }
            }
            off.push_back(sc.size());
            for (size_t j = 0; j < m; j++) {
                sc.push_back(S.s_bl[j]); idx.push_back(gens.slot_B_blinding());
                for (size_t i = 0; i < n; i++) { sc.push_back(S.sL[j * n + i]); idx.push_back(gens.slot_G(j, i)); }
                for (size_t i = 0; i < n; i++) { sc.push_back(S.sR[j * n + i]); idx.push_back(gens.slot_H(j, i)); }
            }
            off.push_back(sc.size());
        });
        std::vector<uint8_t> out;
        if (!run_requests(dev, gens, secret_indexed_msm, reqs, st, out)) return;
        for (size_t p = 0; p < B; p++) {
            if (!st[p].live) continue;
            RangeProofJob &J = jobs[p]; size_t m = st[p].m; const uint8_t *o = out.data() + 32 * st[p].out_base;
            J.commitments.resize(m);
            for (size_t j = 0; j < m; j++) memcpy(J.commitments[j].data(), o + 32 * j, 32);
            memcpy(J.proof.A.data(), o + 32 * m, 32); memcpy(J.proof.S.data(), o + 32 * (m + 1), 32);
        }
    }
    // ---- phase 2: bit challenge, polynomial commitments
    {
        std::vector<MsmReq> reqs(B);
        parallel_for(B, [&](size_t p) {
            if (!st[p].live) return;
            RangeProofJob &J = jobs[p]; ProverState &S = st[p]; size_t m = S.m, N = S.N; Transcript &t = *J.t;
            std::vector<Scalar> &sc = reqs[p].sc; std::vector<uint32_t> &idx = reqs[p].idx; std::vector<uint64_t> &off = reqs[p].off;
            for (size_t j = 0; j < m; j++) t.append_point("V", J.commitments[j]);                        // dealer.rs:107-119
            t.append_point("A", J.proof.A); t.append_point("S", J.proof.S);
            S.y = t.challenge_scalar("y"); S.z = t.challenge_scalar("z"); S.zz = S.z * S.z;
            // party.rs:182-237
            S.l0.resize(N); S.l1.resize(N); S.r0.resize(N); S.r1.resize(N); S.t0.resize(m); S.t1.resize(m); S.t2.resize(m); S.t1_bl.resize(m); S.t2_bl.resize(m); S.offset_zz.resize(m);
            for (size_t j = 0; j < m; j++) {
                Scalar offset_y = scalar_exp_vartime(S.y, (uint64_t)(j * n)), offset_z = scalar_exp_vartime(S.z, (uint64_t)j);
                S.offset_zz[j] = S.zz * offset_z;
                Scalar exp_y = offset_y, exp_2 = Scalar::one();
                for (size_t i = 0; i < n; i++) {
                    size_t q = j * n + i;
                    Scalar a_L = Scalar::from_u64((J.values[j] >> i) & 1), a_R = a_L - one;
                    S.l0[q] = a_L - S.z; S.l1[q] = S.sL[q];
                    S.r0[q] = exp_y * (a_R + S.z) + S.offset_zz[j] * exp_2; S.r1[q] = exp_y * S.sR[q];
                    exp_y *= S.y; exp_2 = exp_2 + exp_2;
                }
                // VecPoly1::inner_product, Karatsuba (util.rs:86-100)
                Scalar acc0 = Scalar::zero(), acc2 = Scalar::zero(), acc1 = Scalar::zero();
                for (size_t i = 0; i < n; i++) { size_t q = j * n + i; acc0 += S.l0[q] * S.r0[q]; acc2 += S.l1[q] * S.r1[q]; acc1 += (S.l0[q] + S.l1[q]) * (S.r0[q] + S.r1[q]); }
                S.t0[j] = acc0; S.t2[j] = acc2; S.t1[j] = acc1 - acc0 - acc2;
            }
            for (size_t j = 0; j < m; j++) { S.t1_bl[j] = Scalar::random(*J.rng); S.t2_bl[j] = Scalar::random(*J.rng); }      // party.rs:214-215, all parties in turn (mod.rs:272-275)
            // T_1 = sum_j (t1_j B + t~1_j B~), T_2 likewise (party.rs:216-217, dealer.rs:169-170)
            for (size_t j = 0; j < m; j++) { sc.push_back(S.t1[j]); idx.push_back(gens.slot_B()); sc.push_back(S.t1_bl[j]); idx.push_back(gens.slot_B_blinding()); }
            off.push_back(sc.size());
            for (size_t j = 0; j < m; j++) { sc.push_back(S.t2[j]); idx.push_back(gens.slot_B()); sc.push_back(S.t2_bl[j]); idx.push_back(gens.slot_B_blinding()); }
            off.push_back(sc.size());
        });
        std::vector<uint8_t> out;
        if (!run_requests(dev, gens, secret_indexed_msm, reqs, st, out)) return;
        for (size_t p = 0; p < B; p++) {
            if (!st[p].live) continue;
            memcpy(jobs[p].proof.T_1.data(), out.data() + 32 * st[p].out_base, 32); memcpy(jobs[p].proof.T_2.data(), out.data() + 32 * (st[p].out_base + 1), 32);
        }
    }
    // ---- phase 3: poly challenge, proof shares, Q = w B
    {
        std::vector<MsmReq> reqs(B);
        parallel_for(B, [&](size_t p) {
            if (!st[p].live) return;
            RangeProofJob &J = jobs[p]; ProverState &S = st[p]; size_t m = S.m, N = S.N; Transcript &t = *J.t; RangeProof &proof = J.proof;
            std::vector<Scalar> &sc = reqs[p].sc; std::vector<uint32_t> &idx = reqs[p].idx; std::vector<uint64_t> &off = reqs[p].off;
            t.append_point("T_1", proof.T_1); t.append_point("T_2", proof.T_2);                          // dealer.rs:172-173
            S.x = t.challenge_scalar("x");
            if (S.x.is_zero()) { J.error = ProofError::MaliciousDealer; S.live = false; return; }        // party.rs:282-284
            // party.rs:279-305, dealer.rs:245-270
            proof.t_x = Scalar::zero(); proof.t_x_blinding = Scalar::zero(); proof.e_blinding = Scalar::zero();
            S.l_vec.resize(N); S.r_vec.resize(N);
            for (size_t j = 0; j < m; j++) {
                proof.t_x += S.t0[j] + S.x * (S.t1[j] + S.x * S.t2[j]);
                proof.t_x_blinding += S.offset_zz[j] * J.blindings[j] + S.x * (S.t1_bl[j] + S.x * S.t2_bl[j]);
                proof.e_blinding += S.a_bl[j] + S.s_bl[j] * S.x;
                for (size_t i = 0; i < n; i++) { size_t q = j * n + i; S.l_vec[q] = S.l0[q] + S.l1[q] * S.x; S.r_vec[q] = S.r0[q] + S.r1[q] * S.x; }
            }
            t.append_scalar("t_x", proof.t_x); t.append_scalar("t_x_blinding", proof.t_x_blinding); t.append_scalar("e_blinding", proof.e_blinding);
            S.w = t.challenge_scalar("w");
            sc.push_back(S.w); idx.push_back(gens.slot_B()); off.push_back(sc.size());                    // Q = w * B (dealer.rs:256)
            S.Gf.assign(N, Scalar::one()); S.Hf.resize(N);
            Scalar y_inv = S.y.invert(), e = Scalar::one();
            for (size_t i = 0; i < N; i++) { S.Hf[i] = e; e *= y_inv; }                                   // dealer.rs:258-261
        });
        std::vector<uint8_t> out;
        if (!run_requests(dev, gens, indexed_msm_vartime, reqs, st, out)) return;          // w is a public challenge (dealer.rs:256)
        for (size_t p = 0; p < B; p++) if (st[p].live) memcpy(st[p].Q.data(), out.data() + 32 * st[p].out_base, 32);
    }
    // ---- phase 4: the inner-product arguments, grouped by aggregation size (one device session per distinct m)
    for (size_t p0 = 0; p0 < B; p0++) {
        if (!st[p0].live) continue;
        size_t m = st[p0].m;
        std::vector<size_t> who; std::vector<Transcript *> ts; std::vector<CompressedRistretto> Qs; std::vector<std::vector<Scalar>> Gfs, Hfs, as, bs;
        for (size_t p = p0; p < B; p++)
            if (st[p].live && st[p].m == m) {
                who.push_back(p); ts.push_back(jobs[p].t); Qs.push_back(st[p].Q); Gfs.push_back(std::move(st[p].Gf)); Hfs.push_back(std::move(st[p].Hf));
                as.push_back(std::move(st[p].l_vec)); bs.push_back(std::move(st[p].r_vec)); st[p].live = false;
            }
        std::vector<InnerProductProof> ipps = InnerProductProof::create_many(dev, gens, n, m, ts, Qs, Gfs, Hfs, as, bs);      // dealer.rs:272-281
        for (size_t k = 0; k < who.size(); k++) jobs[who[k]].proof.ipp_proof = std::move(ipps[k]);
    }
}

ProofError RangeProof::prove_multiple_with_rng(Device &dev, const BulletproofGens &gens, Transcript &t, const std::vector<uint64_t> &values,
                                               const std::vector<Scalar> &blindings, size_t n, Rng &rng, RangeProof &proof, std::vector<CompressedRistretto> &commitments) {
    std::vector<RangeProofJob> jobs(1);
    jobs[0].t = &t; jobs[0].values = values; jobs[0].blindings = blindings; jobs[0].rng = &rng;
    prove_many(dev, gens, n, jobs);
    if (jobs[0].error != ProofError::Ok) return jobs[0].error;
    proof = std::move(jobs[0].proof); commitments = std::move(jobs[0].commitments);
    return ProofError::Ok;
}

ProofError RangeProof::verify_multiple(Device &dev, const BulletproofGens &gens, const Transcript &t, const std::vector<CompressedRistretto> &commitments, size_t n) const {
    std::vector<uint8_t> bytes = to_bytes();
    uint8_t wire[BP_TRANSCRIPT_BYTES]; t.to_wire(wire);
    uint8_t verdict = 0;
    std::vector<uint8_t> vs(32 * commitments.size());
    for (size_t j = 0; j < commitments.size(); j++) memcpy(vs.data() + 32 * j, commitments[j].data(), 32);
    check(bp_rangeproof_verify_batch(dev.ctx, gens.handle, wire, bytes.data(), bytes.size(), vs.data(), n, commitments.size(), 1, nullptr, &verdict), dev.ctx, "bp_rangeproof_verify_batch");
    return (ProofError)verdict;
}

std::vector<uint8_t> RangeProof::to_bytes() const {
    std::vector<uint8_t> buf;
    for (const CompressedRistretto *p : {&A, &S, &T_1, &T_2}) buf.insert(buf.end(), p->begin(), p->end());
    for (const Scalar *s : {&t_x, &t_x_blinding, &e_blinding}) { Bytes32 b = s->to_bytes(); buf.insert(buf.end(), b.begin(), b.end()); }
    std::vector<uint8_t> ipp = ipp_proof.to_bytes(); buf.insert(buf.end(), ipp.begin(), ipp.end());
    return buf;
}
ProofError RangeProof::from_bytes(const uint8_t *s, size_t len, RangeProof &out) {
    if (len % 32 != 0 || len < 7 * 32) return ProofError::FormatError;
    memcpy(out.A.data(), s, 32); memcpy(out.S.data(), s + 32, 32); memcpy(out.T_1.data(), s + 64, 32); memcpy(out.T_2.data(), s + 96, 32);
    if (!Scalar::from_canonical_bytes(s + 128, out.t_x) || !Scalar::from_canonical_bytes(s + 160, out.t_x_blinding) || !Scalar::from_canonical_bytes(s + 192, out.e_blinding)) return ProofError::FormatError;
    return InnerProductProof::from_bytes(s + 224, len - 224, out.ipp_proof);
}

}  // namespace bulletproofs

// ================================================================================================ C shim for the Python harness
using namespace bulletproofs;
extern "C" {

// RangeProof::prove_multiple_with_rng with rng = ChaChaRng::from_seed(rng_seed); transcript is the 203-byte wire state (in: initial, out: final)
int bph_rangeproof_prove(bp_ctx *ctx, bp_gens *gens, size_t gens_capacity, size_t party_capacity, uint8_t *transcript, const uint64_t *values, const uint8_t *blindings,
                         size_t m, size_t n, const uint8_t rng_seed[32], uint8_t *proof_out, uint8_t *commitments_out) {
    try {
        Device dev(ctx); BulletproofGens g{gens, gens_capacity, party_capacity};
        Transcript t(transcript); ChaChaRng rng(rng_seed);
        std::vector<uint64_t> v(values, values + m); std::vector<Scalar> bl(m);
        for (size_t j = 0; j < m; j++) if (!Scalar::from_canonical_bytes(blindings + 32 * j, bl[j])) return -3;
        RangeProof proof; std::vector<CompressedRistretto> V;
        ProofError e = RangeProof::prove_multiple_with_rng(dev, g, t, v, bl, n, rng, proof, V);
        if (e != ProofError::Ok) return (int)e;
        std::vector<uint8_t> bytes = proof.to_bytes();
        memcpy(proof_out, bytes.data(), bytes.size());
        for (size_t j = 0; j < m; j++) memcpy(commitments_out + 32 * j, V[j].data(), 32);
        t.to_wire(transcript);
        return 0;
    } catch (const std::exception &) { return -1; }
}
// B proofs with m values each, every group operation batched across the proofs: transcripts all start from `transcript`, proof p uses
// ChaChaRng::from_seed(rng_seeds[p]); status_out[p] = ProofError code
int bph_rangeproof_prove_many(bp_ctx *ctx, bp_gens *gens, size_t gens_capacity, size_t party_capacity, const uint8_t *transcript, const uint64_t *values, const uint8_t *blindings,
                              size_t m, size_t n, size_t count, const uint8_t *rng_seeds, uint8_t *proofs_out, size_t proof_len, uint8_t *commitments_out, uint8_t *status_out) {
    try {
        Device dev(ctx); BulletproofGens g{gens, gens_capacity, party_capacity};
        std::vector<Transcript> ts(count, Transcript(transcript)); std::vector<ChaChaRng> rngs; rngs.reserve(count);
        std::vector<RangeProofJob> jobs(count);
        for (size_t p = 0; p < count; p++) {
            rngs.emplace_back(rng_seeds + 32 * p);
            jobs[p].t = &ts[p]; jobs[p].rng = &rngs[p];
            jobs[p].values.assign(values + p * m, values + (p + 1) * m); jobs[p].blindings.resize(m);
            for (size_t j = 0; j < m; j++) if (!Scalar::from_canonical_bytes(blindings + 32 * (p * m + j), jobs[p].blindings[j])) return -3;
        }
        RangeProof::prove_many(dev, g, n, jobs);
        for (size_t p = 0; p < count; p++) {
            status_out[p] = (uint8_t)jobs[p].error;
            if (jobs[p].error != ProofError::Ok) continue;
            std::vector<uint8_t> bytes = jobs[p].proof.to_bytes();
            if (bytes.size() != proof_len) return -4;
            memcpy(proofs_out + p * proof_len, bytes.data(), proof_len);
            for (size_t j = 0; j < m; j++) memcpy(commitments_out + 32 * (p * m + j), jobs[p].commitments[j].data(), 32);
        }
        return 0;
    } catch (const std::exception &) { return -1; }
}
// RangeProof::from_bytes + verify_multiple
int bph_rangeproof_verify(bp_ctx *ctx, bp_gens *gens, size_t gens_capacity, size_t party_capacity, const uint8_t *transcript, const uint8_t *proof, size_t proof_len,
                          const uint8_t *commitments, size_t m, size_t n) {
    try {
        Device dev(ctx); BulletproofGens g{gens, gens_capacity, party_capacity};
        RangeProof p; ProofError e = RangeProof::from_bytes(proof, proof_len, p);
        if (e != ProofError::Ok) return (int)e;
        std::vector<CompressedRistretto> V(m); for (size_t j = 0; j < m; j++) memcpy(V[j].data(), commitments + 32 * j, 32);
        return (int)p.verify_multiple(dev, g, Transcript(transcript), V, n);
    } catch (const std::exception &) { return -1; }
}
static bool load_scalars(const uint8_t *b, size_t n, std::vector<Scalar> &out);
static std::vector<CompressedRistretto> load_points(const uint8_t *b, size_t n);
// LinearProof::create with rng = ChaChaRng::from_seed(seed); proof_out = 32*(2 lg n + 3) bytes
int bph_linear_create(bp_ctx *ctx, uint8_t *transcript, const uint8_t seed[32], const uint8_t C[32], const uint8_t r[32], const uint8_t *a, const uint8_t *b, const uint8_t *G,
                      const uint8_t F[32], const uint8_t B[32], size_t n, uint8_t *proof_out) {
    try {
        Device dev(ctx); Transcript t(transcript); ChaChaRng rng(seed);
        std::vector<Scalar> av, bv; Scalar rr;
        if (!load_scalars(a, n, av) || !load_scalars(b, n, bv) || !Scalar::from_canonical_bytes(r, rr)) return -3;
        CompressedRistretto c, f, bb; memcpy(c.data(), C, 32); memcpy(f.data(), F, 32); memcpy(bb.data(), B, 32);
        LinearProof p; ProofError e = LinearProof::create(dev, t, rng, c, rr, av, bv, load_points(G, n), f, bb, p);
        if (e != ProofError::Ok) return (int)e;
        std::vector<uint8_t> bytes = p.to_bytes(); memcpy(proof_out, bytes.data(), bytes.size());
        t.to_wire(transcript);
        return 0;
    } catch (const std::exception &) { return -1; }
}
int bph_linear_verify(bp_ctx *ctx, uint8_t *transcript, const uint8_t *proof, size_t proof_len, const uint8_t C[32], const uint8_t *G, const uint8_t F[32], const uint8_t B[32],
                      const uint8_t *b, size_t n) {
    try {
        Device dev(ctx); Transcript t(transcript);
        LinearProof p; ProofError e = LinearProof::from_bytes(proof, proof_len, p);
        if (e != ProofError::Ok) return (int)e;
        std::vector<Scalar> bv; if (!load_scalars(b, n, bv)) return -3;
        CompressedRistretto c, f, bb; memcpy(c.data(), C, 32); memcpy(f.data(), F, 32); memcpy(bb.data(), B, 32);
        e = p.verify(dev, t, c, load_points(G, n), f, bb, bv);
        t.to_wire(transcript);
        return (int)e;
    } catch (const std::exception &) { return -1; }
}
static bool load_scalars(const uint8_t *b, size_t n, std::vector<Scalar> &out) { out.resize(n); for (size_t i = 0; i < n; i++) if (!Scalar::from_canonical_bytes(b + 32 * i, out[i])) return false; return true; }
static std::vector<CompressedRistretto> load_points(const uint8_t *b, size_t n) { std::vector<CompressedRistretto> v(n); for (size_t i = 0; i < n; i++) memcpy(v[i].data(), b + 32 * i, 32); return v; }
// InnerProductProof::create over arbitrary compressed vectors; proof_out = 32*(2 lg n + 2) bytes
int bph_ipp_create(bp_ctx *ctx, uint8_t *transcript, const uint8_t Q[32], const uint8_t *Gf, const uint8_t *Hf, const uint8_t *G, const uint8_t *H,
                   const uint8_t *a, const uint8_t *b, size_t n, uint8_t *proof_out) {
    try {
        Device dev(ctx); Transcript t(transcript);
        std::vector<Scalar> gf, hf, av, bv;
        if (!load_scalars(Gf, n, gf) || !load_scalars(Hf, n, hf) || !load_scalars(a, n, av) || !load_scalars(b, n, bv)) return -3;
        CompressedRistretto q; memcpy(q.data(), Q, 32);
        InnerProductProof p = InnerProductProof::create(dev, t, q, gf, hf, load_points(G, n), load_points(H, n), av, bv);
        std::vector<uint8_t> bytes = p.to_bytes(); memcpy(proof_out, bytes.data(), bytes.size());
        t.to_wire(transcript);
        return 0;
    } catch (const std::exception &) { return -1; }
}
int bph_ipp_verify(bp_ctx *ctx, uint8_t *transcript, size_t n, const uint8_t *Gf, const uint8_t *Hf, const uint8_t P[32], const uint8_t Q[32],
                   const uint8_t *G, const uint8_t *H, const uint8_t *proof, size_t proof_len) {
    try {
        Device dev(ctx); Transcript t(transcript);
        InnerProductProof p; ProofError e = InnerProductProof::from_bytes(proof, proof_len, p);
        if (e != ProofError::Ok) return (int)e;
        std::vector<Scalar> gf, hf; if (!load_scalars(Gf, n, gf) || !load_scalars(Hf, n, hf)) return -3;
        CompressedRistretto pp, q; memcpy(pp.data(), P, 32); memcpy(q.data(), Q, 32);
        e = p.verify(dev, n, t, gf, hf, pp, q, load_points(G, n), load_points(H, n));
        t.to_wire(transcript);
        return (int)e;
    } catch (const std::exception &) { return -1; }
}
}
