// Host mirror of the reference's r1cs module (see r1cs.hpp).  Scalars and transcripts on the host, every MSM on the GPU.
#include "r1cs.hpp"

namespace bulletproofs {
namespace r1cs {

static void check(int rc, bp_ctx *ctx, const char *what) {
    if (rc != BP_OK) throw std::runtime_error(std::string(what) + " failed with code " + std::to_string(rc) + ": " + bp_last_error(ctx));
}
static std::vector<uint8_t> pack(const std::vector<Scalar> &v) {
    std::vector<uint8_t> o(32 * v.size());
    const size_t CH = 8192, nch = (v.size() + CH - 1) / CH;
    parallel_for(nch, [&](size_t c) { for (size_t i = c * CH; i < std::min(v.size(), (c + 1) * CH); i++) v[i].write(o.data() + 32 * i); });
    return o;
}
static size_t next_pow2(size_t n) { size_t p = 1; while (p < n) p <<= 1; return p; }
static bool is_identity(const CompressedRistretto &p) { uint8_t z = 0; for (uint8_t b : p) z |= b; return z == 0; }

// ------------------------------------------------------------------ TranscriptRng
TranscriptRng::TranscriptRng(const Transcript &t) { uint8_t wire[BP_TRANSCRIPT_BYTES]; t.to_wire(wire); m_.st = st_; merlin_load(m_, wire); }
void TranscriptRng::rekey_with_witness_bytes(const char *label, const uint8_t *w, size_t len) {
    uint32_t ll = 0; while (label[ll]) ll++;
    uint8_t l4[4] = {(uint8_t)len, (uint8_t)(len >> 8), (uint8_t)(len >> 16), (uint8_t)(len >> 24)};
    strobe_begin_op(m_, 16 | 2); strobe_absorb(m_, (const uint8_t *)label, ll); strobe_absorb(m_, l4, 4);      // meta_ad(label), meta_ad(len, more)
    strobe_begin_op(m_, 2 | 4); strobe_overwrite(m_, w, (uint32_t)len);                                            // key(witness)
}
void TranscriptRng::finalize(Rng &external) {
    uint8_t rb[32]; external.fill_bytes(rb, 32);
    strobe_begin_op(m_, 16 | 2); strobe_absorb(m_, (const uint8_t *)"rng", 3);
    strobe_begin_op(m_, 2 | 4); strobe_overwrite(m_, rb, 32);
}
void TranscriptRng::fill_bytes(uint8_t *out, size_t n) {
    uint8_t l4[4] = {(uint8_t)n, (uint8_t)(n >> 8), (uint8_t)(n >> 16), (uint8_t)(n >> 24)};
    strobe_begin_op(m_, 16 | 2); strobe_absorb(m_, l4, 4);
    strobe_begin_op(m_, 1 | 2 | 4); strobe_squeeze(m_, out, (uint32_t)n);
}

// ------------------------------------------------------------------ R1CSProof wire format (proof.rs:83-204)
std::vector<uint8_t> R1CSProof::to_bytes() const {
    std::vector<uint8_t> buf;
    bool one_phase = is_identity(A_I2) && is_identity(A_O2) && is_identity(S2);
    buf.push_back(one_phase ? 0 : 1);
    auto put = [&](const CompressedRistretto &p) { buf.insert(buf.end(), p.begin(), p.end()); };
    put(A_I1); put(A_O1); put(S1);
    if (!one_phase) { put(A_I2); put(A_O2); put(S2); }
    put(T_1); put(T_3); put(T_4); put(T_5); put(T_6);
    put(t_x.to_bytes()); put(t_x_blinding.to_bytes()); put(e_blinding.to_bytes());
    std::vector<uint8_t> ipp = ipp_proof.to_bytes(); buf.insert(buf.end(), ipp.begin(), ipp.end());
    return buf;
}
R1CSError R1CSProof::from_bytes(const uint8_t *s, size_t len, R1CSProof &out) {
    if (len < 1) return R1CSError::FormatError;
    uint8_t version = s[0]; s++; len--;
    if (len % 32 != 0) return R1CSError::FormatError;
    size_t minlen = version == 0 ? 11 * 32 : version == 1 ? 14 * 32 : 0;
    if (!minlen || len < minlen) return R1CSError::FormatError;
    auto get = [&](CompressedRistretto &p) { memcpy(p.data(), s, 32); s += 32; len -= 32; };
    get(out.A_I1); get(out.A_O1); get(out.S1);
    if (version == 1) { get(out.A_I2); get(out.A_O2); get(out.S2); } else { out.A_I2.fill(0); out.A_O2.fill(0); out.S2.fill(0); }
    get(out.T_1); get(out.T_3); get(out.T_4); get(out.T_5); get(out.T_6);
    if (!Scalar::from_canonical_bytes(s, out.t_x) || !Scalar::from_canonical_bytes(s + 32, out.t_x_blinding) || !Scalar::from_canonical_bytes(s + 64, out.e_blinding)) return R1CSError::FormatError;
    s += 96; len -= 96;
    return InnerProductProof::from_bytes(s, len, out.ipp_proof) == ProofError::Ok ? R1CSError::Ok : R1CSError::FormatError;
}

// ------------------------------------------------------------------ flattened constraints (prover.rs:301-338, verifier.rs:260-298)
static void flatten(const std::vector<LinearCombination> &constraints, const Scalar &z, size_t n, size_t m,
                    std::vector<Scalar> &wL, std::vector<Scalar> &wR, std::vector<Scalar> &wO, std::vector<Scalar> &wV, Scalar &wc) {
    wL.assign(n, Scalar::zero()); wR.assign(n, Scalar::zero()); wO.assign(n, Scalar::zero()); wV.assign(m, Scalar::zero()); wc = Scalar::zero();
    Scalar exp_z = z;
    for (const LinearCombination &lc : constraints) {
        for (const auto &term : lc.terms) {
            Scalar c = exp_z * term.second; size_t i = term.first.index;
            switch (term.first.kind) {
                case VarKind::MultiplierLeft: wL[i] += c; break;
                case VarKind::MultiplierRight: wR[i] += c; break;
                case VarKind::MultiplierOutput: wO[i] += c; break;
                case VarKind::Committed: wV[i] = wV[i] - c; break;
                case VarKind::One: wc = wc - c; break;
            }
        }
        exp_z *= z;
    }
}

// ------------------------------------------------------------------ Prover
Prover::Prover(Device &dev, const BulletproofGens &gens, Transcript &t) : t_(t), gens_(gens), dev_(dev) {
    t_.append_message("dom-sep", (const uint8_t *)"r1cs v1", 7);                       // transcript.rs:55-57
}
std::pair<CompressedRistretto, Variable> Prover::commit(const Scalar &v, const Scalar &v_blinding) {
    size_t i = v_.size(); v_.push_back(v); v_blinding_.push_back(v_blinding);
    // PedersenGens::commit (generators.rs:39-41) on the GPU
    std::vector<Scalar> sc = {v, v_blinding}; uint32_t idx[2] = {gens_.slot_B(), gens_.slot_B_blinding()}; uint64_t off[2] = {0, 2}; uint8_t st;
    CompressedRistretto V;
    check(secret_indexed_msm(dev_.ctx, gens_.handle, pack(sc).data(), idx, off, 1, V.data(), &st), dev_.ctx, "commit");
    t_.append_point("V", V);
    return {V, Variable{VarKind::Committed, i}};
}
std::vector<std::pair<CompressedRistretto, Variable>> Prover::commit_vec(const std::vector<Scalar> &v, const std::vector<Scalar> &v_blinding) {
    if (v.size() != v_blinding.size()) throw std::invalid_argument("commit_vec: lengths differ");
    size_t m = v.size();
    std::vector<std::pair<CompressedRistretto, Variable>> out(m);
    if (m == 0) return out;
    std::vector<Scalar> sc(2 * m); std::vector<uint32_t> idx(2 * m); std::vector<uint64_t> off(m + 1); std::vector<uint8_t> outs(32 * m), st(m);
    for (size_t i = 0; i < m; i++) { sc[2 * i] = v[i]; sc[2 * i + 1] = v_blinding[i]; idx[2 * i] = gens_.slot_B(); idx[2 * i + 1] = gens_.slot_B_blinding(); off[i] = 2 * i; }
    off[m] = 2 * m;
    check(secret_indexed_msm(dev_.ctx, gens_.handle, pack(sc).data(), idx.data(), off.data(), m, outs.data(), st.data()), dev_.ctx, "commit_vec");
    for (size_t i = 0; i < m; i++) {
        size_t j = v_.size(); v_.push_back(v[i]); v_blinding_.push_back(v_blinding[i]);
        memcpy(out[i].first.data(), outs.data() + 32 * i, 32); out[i].second = Variable{VarKind::Committed, j};
        t_.append_point("V", out[i].first);
    }
    return out;
}
Scalar Prover::eval(const LinearCombination &lc) const {
    Scalar acc = Scalar::zero();
    for (const auto &term : lc.terms) {
        Scalar val;
        switch (term.first.kind) {
            case VarKind::MultiplierLeft: val = a_L_[term.first.index]; break;
            case VarKind::MultiplierRight: val = a_R_[term.first.index]; break;
            case VarKind::MultiplierOutput: val = a_O_[term.first.index]; break;
            case VarKind::Committed: val = v_[term.first.index]; break;
            default: val = Scalar::one();
        }
        acc += term.second * val;
    }
    return acc;
}
Multiplier Prover::multiply(LinearCombination left, LinearCombination right) {           // prover.rs:73-103
    Scalar l = eval(left), r = eval(right), o = l * r;
    size_t i = a_L_.size();
    Multiplier mv{{VarKind::MultiplierLeft, i}, {VarKind::MultiplierRight, i}, {VarKind::MultiplierOutput, i}};
    a_L_.push_back(l); a_R_.push_back(r); a_O_.push_back(o);
    left.terms.push_back({mv.left, -Scalar::one()}); right.terms.push_back({mv.right, -Scalar::one()});
    constrain(std::move(left)); constrain(std::move(right));
    return mv;
}
R1CSError Prover::allocate(const Scalar *assignment, Variable &out) {                    // prover.rs:105-126
    if (!assignment) return R1CSError::MissingAssignment;
    if (!pending_) { size_t i = a_L_.size(); pending_ = true; pending_idx_ = i; a_L_.push_back(*assignment); a_R_.push_back(Scalar::zero()); a_O_.push_back(Scalar::zero()); out = {VarKind::MultiplierLeft, i}; }
    else { size_t i = pending_idx_; pending_ = false; a_R_[i] = *assignment; a_O_[i] = a_L_[i] * a_R_[i]; out = {VarKind::MultiplierRight, i}; }
    return R1CSError::Ok;
}
R1CSError Prover::allocate_multiplier(const std::pair<Scalar, Scalar> *a, Multiplier &out) {   // prover.rs:128-146
    if (!a) return R1CSError::MissingAssignment;
    size_t i = a_L_.size();
    a_L_.push_back(a->first); a_R_.push_back(a->second); a_O_.push_back(a->first * a->second);
    out = Multiplier{{VarKind::MultiplierLeft, i}, {VarKind::MultiplierRight, i}, {VarKind::MultiplierOutput, i}};
    return R1CSError::Ok;
}

// blinding * B~ + <a, G[g0..)> + <b, H[g0..)> as one indexed MSM term list
static void push_vector_commitment(std::vector<Scalar> &sc, std::vector<uint32_t> &idx, std::vector<uint64_t> &off, const BulletproofGens &g, const Scalar &blinding,
                                   const Scalar *a, const Scalar *b, size_t g0, size_t count) {
    sc.push_back(blinding); idx.push_back(g.slot_B_blinding());
    for (size_t i = 0; i < count; i++) { sc.push_back(a[i]); idx.push_back(g.slot_G(0, g0 + i)); }
    if (b) for (size_t i = 0; i < count; i++) { sc.push_back(b[i]); idx.push_back(g.slot_H(0, g0 + i)); }
    off.push_back(sc.size());
}

R1CSError Prover::prove(Rng &external_rng, R1CSProof &proof) {
    t_.append_u64("m", (uint64_t)v_.size());
    TranscriptRng rng(t_);                                                                // prover.rs:403-413
    for (const Scalar &vb : v_blinding_) { Bytes32 b = vb.to_bytes(); rng.rekey_with_witness_bytes("v_blinding", b.data(), 32); }
    rng.finalize(external_rng);
    size_t n1 = a_L_.size();
    if (gens_.gens_capacity < n1) return R1CSError::InvalidGeneratorsLength;
    Scalar i_bl1 = Scalar::random(rng), o_bl1 = Scalar::random(rng), s_bl1 = Scalar::random(rng);
    std::vector<Scalar> s_L(n1), s_R(n1);
    for (size_t i = 0; i < n1; i++) s_L[i] = Scalar::random(rng);
    for (size_t i = 0; i < n1; i++) s_R[i] = Scalar::random(rng);
    {   // A_I1, A_O1, S1: three MSMs over [B~ | G | H] in one call (prover.rs:433-459)
        std::vector<Scalar> sc; std::vector<uint32_t> idx; std::vector<uint64_t> off = {0};
        push_vector_commitment(sc, idx, off, gens_, i_bl1, a_L_.data(), a_R_.data(), 0, n1);
        push_vector_commitment(sc, idx, off, gens_, o_bl1, a_O_.data(), nullptr, 0, n1);
        push_vector_commitment(sc, idx, off, gens_, s_bl1, s_L.data(), s_R.data(), 0, n1);
        uint8_t out[96], st[3];
        check(secret_indexed_msm(dev_.ctx, gens_.handle, pack(sc).data(), idx.data(), off.data(), 3, out, st), dev_.ctx, "phase-1 commitments");
        memcpy(proof.A_I1.data(), out, 32); memcpy(proof.A_O1.data(), out + 32, 32); memcpy(proof.S1.data(), out + 64, 32);
    }
    t_.append_point("A_I1", proof.A_I1); t_.append_point("A_O1", proof.A_O1); t_.append_point("S1", proof.S1);
    // create_randomized_constraints (prover.rs:358-377)
    pending_ = false;
    if (deferred_.empty()) t_.append_message("dom-sep", (const uint8_t *)"r1cs-1phase", 11);
    else {
        t_.append_message("dom-sep", (const uint8_t *)"r1cs-2phase", 11);
        std::vector<Callback> cbs = std::move(deferred_); deferred_.clear();
        for (auto &cb : cbs) { R1CSError e = cb(*this); if (e != R1CSError::Ok) return e; }
    }
    size_t n = a_L_.size(), n2 = n - n1, padded_n = next_pow2(n);
    if (gens_.gens_capacity < padded_n) return R1CSError::InvalidGeneratorsLength;
    Scalar i_bl2, o_bl2, s_bl2;
    if (n2 > 0) { i_bl2 = Scalar::random(rng); o_bl2 = Scalar::random(rng); s_bl2 = Scalar::random(rng); }
    s_L.resize(n); s_R.resize(n);
    for (size_t i = n1; i < n; i++) s_L[i] = Scalar::random(rng);
    for (size_t i = n1; i < n; i++) s_R[i] = Scalar::random(rng);
    proof.A_I2.fill(0); proof.A_O2.fill(0); proof.S2.fill(0);
    if (n2 > 0) {                                                                        // prover.rs:500-524
        std::vector<Scalar> sc; std::vector<uint32_t> idx; std::vector<uint64_t> off = {0};
        push_vector_commitment(sc, idx, off, gens_, i_bl2, a_L_.data() + n1, a_R_.data() + n1, n1, n2);
        push_vector_commitment(sc, idx, off, gens_, o_bl2, a_O_.data() + n1, nullptr, n1, n2);
        push_vector_commitment(sc, idx, off, gens_, s_bl2, s_L.data() + n1, s_R.data() + n1, n1, n2);
        uint8_t out[96], st[3];
        check(secret_indexed_msm(dev_.ctx, gens_.handle, pack(sc).data(), idx.data(), off.data(), 3, out, st), dev_.ctx, "phase-2 commitments");
        memcpy(proof.A_I2.data(), out, 32); memcpy(proof.A_O2.data(), out + 32, 32); memcpy(proof.S2.data(), out + 64, 32);
    }
    t_.append_point("A_I2", proof.A_I2); t_.append_point("A_O2", proof.A_O2); t_.append_point("S2", proof.S2);
    Scalar y = t_.challenge_scalar("y"), z = t_.challenge_scalar("z");
    std::vector<Scalar> wL, wR, wO, wV; Scalar wc;
    flatten(constraints_, z, n, v_.size(), wL, wR, wO, wV, wc);
    // l(x), r(x) (prover.rs:547-573) and t(x) = <l, r> (util.rs:125-142)
    std::vector<Scalar> l1(n), l2(n), l3(n), r0(n), r1(n), r3(n), exp_y_inv(padded_n);
    Scalar y_inv = y.invert(), exp_y = Scalar::one();
    // powers of y and y^-1 and the six coefficient vectors, chunked over the host cores (each chunk starts from its own power)
    const size_t CH = 4096, nch = (padded_n + CH - 1) / CH;
    std::vector<Scalar> exp_y_pow(padded_n);
    parallel_for(nch, [&](size_t c) {
        size_t lo = c * CH, hi = std::min(padded_n, lo + CH);
        Scalar e = scalar_exp_vartime(y_inv, (uint64_t)lo), f = scalar_exp_vartime(y, (uint64_t)lo);
        for (size_t i = lo; i < hi; i++) { exp_y_inv[i] = e; e *= y_inv; exp_y_pow[i] = f; f *= y; }
        for (size_t i = lo; i < std::min(hi, n); i++) {
            l1[i] = a_L_[i] + exp_y_inv[i] * wR[i]; l2[i] = a_O_[i]; l3[i] = s_L[i];
            r0[i] = wO[i] - exp_y_pow[i]; r1[i] = exp_y_pow[i] * a_R_[i] + wL[i]; r3[i] = exp_y_pow[i] * s_R[i];
        }
    });
    (void)exp_y;
    Scalar t1 = inner_product(l1, r0), t2 = inner_product(l1, r1) + inner_product(l2, r0), t3 = inner_product(l2, r1) + inner_product(l3, r0),
           t4 = inner_product(l1, r3) + inner_product(l3, r1), t5 = inner_product(l2, r3), t6 = inner_product(l3, r3);
    Scalar t1b = Scalar::random(rng), t3b = Scalar::random(rng), t4b = Scalar::random(rng), t5b = Scalar::random(rng), t6b = Scalar::random(rng);
    {   // T_1, T_3, T_4, T_5, T_6: five Pedersen commitments in one call (prover.rs:587-591)
        std::vector<Scalar> sc = {t1, t1b, t3, t3b, t4, t4b, t5, t5b, t6, t6b}; std::vector<uint32_t> idx; std::vector<uint64_t> off = {0};
        for (int k = 0; k < 5; k++) { idx.push_back(gens_.slot_B()); idx.push_back(gens_.slot_B_blinding()); off.push_back(2 * (k + 1)); }
        uint8_t out[160], st[5];
        check(secret_indexed_msm(dev_.ctx, gens_.handle, pack(sc).data(), idx.data(), off.data(), 5, out, st), dev_.ctx, "T commitments");
        CompressedRistretto *Ts[5] = {&proof.T_1, &proof.T_3, &proof.T_4, &proof.T_5, &proof.T_6};
        for (int k = 0; k < 5; k++) memcpy(Ts[k]->data(), out + 32 * k, 32);
    }
    t_.append_point("T_1", proof.T_1); t_.append_point("T_3", proof.T_3); t_.append_point("T_4", proof.T_4); t_.append_point("T_5", proof.T_5); t_.append_point("T_6", proof.T_6);
    Scalar u = t_.challenge_scalar("u"), x = t_.challenge_scalar("x");
    Scalar t2b = Scalar::zero();
    for (size_t i = 0; i < v_.size(); i++) t2b += wV[i] * v_blinding_[i];
    proof.t_x = x * (t1 + x * (t2 + x * (t3 + x * (t4 + x * (t5 + x * t6)))));            // Poly6::eval (util.rs:164-168)
    proof.t_x_blinding = x * (t1b + x * (t2b + x * (t3b + x * (t4b + x * (t5b + x * t6b)))));
    std::vector<Scalar> l_vec(padded_n), r_vec(padded_n);
    parallel_for(nch, [&](size_t c) {
        size_t lo = c * CH, hi = std::min(padded_n, lo + CH);
        for (size_t i = lo; i < hi; i++) {
            if (i < n) { l_vec[i] = x * (l1[i] + x * (l2[i] + x * l3[i])); r_vec[i] = r0[i] + x * (r1[i] + x * (x * r3[i])); }
            else r_vec[i] = -exp_y_pow[i];
        }
    });
    Scalar i_bl = i_bl1 + u * i_bl2, o_bl = o_bl1 + u * o_bl2, s_bl = s_bl1 + u * s_bl2;
    proof.e_blinding = x * (i_bl + x * (o_bl + x * s_bl));
    t_.append_scalar("t_x", proof.t_x); t_.append_scalar("t_x_blinding", proof.t_x_blinding); t_.append_scalar("e_blinding", proof.e_blinding);
    Scalar w = t_.challenge_scalar("w");
    CompressedRistretto Q; uint32_t qi = gens_.slot_B(); uint64_t qo[2] = {0, 1}; uint8_t qs;
    check(bp_msm_indexed_batch(dev_.ctx, gens_.handle, w.to_bytes().data(), &qi, nullptr, 0, qo, 1, Q.data(), &qs), dev_.ctx, "Q");     // w is a public challenge: variable-time
    std::vector<Scalar> Gf(padded_n), Hf(padded_n);
    parallel_for(nch, [&](size_t c) {                                                                                 // prover.rs:648-656
        for (size_t i = c * CH; i < std::min(padded_n, (c + 1) * CH); i++) { Gf[i] = i < n1 ? Scalar::one() : u; Hf[i] = exp_y_inv[i] * Gf[i]; }
    });
    proof.ipp_proof = InnerProductProof::create(dev_, gens_, padded_n, 1, t_, Q, Gf, Hf, std::move(l_vec), std::move(r_vec));
    return R1CSError::Ok;
}

// ------------------------------------------------------------------ Verifier
Verifier::Verifier(Device &dev, const BulletproofGens &gens, Transcript &t) : t_(t), gens_(gens), dev_(dev) {
    t_.append_message("dom-sep", (const uint8_t *)"r1cs v1", 7);
}
Variable Verifier::commit(const CompressedRistretto &V) { size_t i = V_.size(); V_.push_back(V); t_.append_point("V", V); return {VarKind::Committed, i}; }
Multiplier Verifier::multiply(LinearCombination left, LinearCombination right) {          // verifier.rs:66-86
    size_t i = num_vars_++;
    Multiplier mv{{VarKind::MultiplierLeft, i}, {VarKind::MultiplierRight, i}, {VarKind::MultiplierOutput, i}};
    left.terms.push_back({mv.left, -Scalar::one()}); right.terms.push_back({mv.right, -Scalar::one()});
    constrain(std::move(left)); constrain(std::move(right));
    return mv;
}
R1CSError Verifier::allocate(const Scalar *, Variable &out) {                             // verifier.rs:88-102
    if (!pending_) { size_t i = num_vars_++; pending_ = true; pending_idx_ = i; out = {VarKind::MultiplierLeft, i}; }
    else { pending_ = false; out = {VarKind::MultiplierRight, pending_idx_}; }
    return R1CSError::Ok;
}
R1CSError Verifier::allocate_multiplier(const std::pair<Scalar, Scalar> *, Multiplier &out) {
    size_t i = num_vars_++;
    out = Multiplier{{VarKind::MultiplierLeft, i}, {VarKind::MultiplierRight, i}, {VarKind::MultiplierOutput, i}};
    return R1CSError::Ok;
}

R1CSError Verifier::verify(const R1CSProof &proof, Rng &external_rng) {
    t_.append_u64("m", (uint64_t)V_.size());
    size_t n1 = num_vars_;
    if (!t_.validate_and_append_point("A_I1", proof.A_I1) || !t_.validate_and_append_point("A_O1", proof.A_O1) || !t_.validate_and_append_point("S1", proof.S1)) return R1CSError::VerificationError;
    pending_ = false;
    if (deferred_.empty()) t_.append_message("dom-sep", (const uint8_t *)"r1cs-1phase", 11);
    else {
        t_.append_message("dom-sep", (const uint8_t *)"r1cs-2phase", 11);
        std::vector<Callback> cbs = std::move(deferred_); deferred_.clear();
        for (auto &cb : cbs) { R1CSError e = cb(*this); if (e != R1CSError::Ok) return e; }
    }
    size_t n = num_vars_, padded_n = next_pow2(n);
    if (gens_.gens_capacity < padded_n) return R1CSError::InvalidGeneratorsLength;
    t_.append_point("A_I2", proof.A_I2); t_.append_point("A_O2", proof.A_O2); t_.append_point("S2", proof.S2);
    Scalar y = t_.challenge_scalar("y"), z = t_.challenge_scalar("z");
    if (!t_.validate_and_append_point("T_1", proof.T_1) || !t_.validate_and_append_point("T_3", proof.T_3) || !t_.validate_and_append_point("T_4", proof.T_4) ||
        !t_.validate_and_append_point("T_5", proof.T_5) || !t_.validate_and_append_point("T_6", proof.T_6)) return R1CSError::VerificationError;
    Scalar u = t_.challenge_scalar("u"), x = t_.challenge_scalar("x");
    t_.append_scalar("t_x", proof.t_x); t_.append_scalar("t_x_blinding", proof.t_x_blinding); t_.append_scalar("e_blinding", proof.e_blinding);
    Scalar w = t_.challenge_scalar("w");
    std::vector<Scalar> wL, wR, wO, wV; Scalar wc;
    flatten(constraints_, z, n, V_.size(), wL, wR, wO, wV, wc);
    std::vector<Scalar> u_sq, u_inv_sq, s;
    if (proof.ipp_proof.verification_scalars(padded_n, t_, u_sq, u_inv_sq, s) != ProofError::Ok) return R1CSError::VerificationError;
    size_t k = proof.ipp_proof.L_vec.size();
    const Scalar &a = proof.ipp_proof.a, &b = proof.ipp_proof.b;
    Scalar y_inv = y.invert();
    std::vector<Scalar> y_inv_vec(padded_n), yneg_wR(padded_n, Scalar::zero());
    { Scalar e = Scalar::one(); for (size_t i = 0; i < padded_n; i++) { y_inv_vec[i] = e; e *= y_inv; } }
    Scalar delta = Scalar::zero();
    for (size_t i = 0; i < n; i++) { yneg_wR[i] = wR[i] * y_inv_vec[i]; delta += yneg_wR[i] * wL[i]; }
    TranscriptRng rng(t_); rng.finalize(external_rng);                                   // verifier.rs:447-449
    Scalar r = Scalar::random(rng), xx = x * x, rxx = r * xx, xxx = x * xx;
    // the mega-check (verifier.rs:459-491): static G/H/B/B~ by table slot, everything else uploaded compressed
    std::vector<Scalar> sc; std::vector<uint32_t> idx; std::vector<uint8_t> dyn;
    auto dyn_term = [&](const Scalar &s_, const CompressedRistretto &p) { sc.push_back(s_); idx.push_back(0x80000000u | (uint32_t)(dyn.size() / 32)); dyn.insert(dyn.end(), p.begin(), p.end()); };
    dyn_term(x, proof.A_I1); dyn_term(xx, proof.A_O1); dyn_term(xxx, proof.S1);
    dyn_term(u * x, proof.A_I2); dyn_term(u * xx, proof.A_O2); dyn_term(u * xxx, proof.S2);
    for (size_t i = 0; i < V_.size(); i++) dyn_term(wV[i] * rxx, V_[i]);
    dyn_term(r * x, proof.T_1); dyn_term(rxx * x, proof.T_3); dyn_term(rxx * xx, proof.T_4); dyn_term(rxx * xxx, proof.T_5); dyn_term(rxx * xx * xx, proof.T_6);
    sc.push_back(w * (proof.t_x - a * b) + r * (xx * (wc + delta) - proof.t_x)); idx.push_back(gens_.slot_B());
    sc.push_back(-proof.e_blinding - r * proof.t_x_blinding); idx.push_back(gens_.slot_B_blinding());
    for (size_t i = 0; i < padded_n; i++) { Scalar u1 = i < n1 ? Scalar::one() : u; sc.push_back(u1 * (x * yneg_wR[i] - a * s[i])); idx.push_back(gens_.slot_G(0, i)); }
    for (size_t i = 0; i < padded_n; i++) {
        Scalar u1 = i < n1 ? Scalar::one() : u, wLi = i < n ? wL[i] : Scalar::zero(), wOi = i < n ? wO[i] : Scalar::zero();
        sc.push_back(u1 * (y_inv_vec[i] * (x * wLi + wOi - b * s[padded_n - 1 - i]) - Scalar::one())); idx.push_back(gens_.slot_H(0, i));
    }
    for (size_t i = 0; i < k; i++) dyn_term(u_sq[i], proof.ipp_proof.L_vec[i]);
    for (size_t i = 0; i < k; i++) dyn_term(u_inv_sq[i], proof.ipp_proof.R_vec[i]);
    uint64_t off[2] = {0, sc.size()}; uint8_t st = 0; CompressedRistretto mega;
    check(bp_msm_indexed_batch(dev_.ctx, gens_.handle, pack(sc).data(), idx.data(), dyn.data(), dyn.size() / 32, off, 1, mega.data(), &st), dev_.ctx, "mega-check");
    if (st == BP_ERR_INVALID_POINT) return R1CSError::VerificationError;                 // optional_multiscalar_mul -> None
    return is_identity(mega) ? R1CSError::Ok : R1CSError::VerificationError;             // is_identity(): the identity coset encodes as zeros
}

// ------------------------------------------------------------------ gadgets
R1CSError shuffle_gadget(ConstraintSystem &cs, std::vector<Variable> x, std::vector<Variable> y) {
    if (x.size() != y.size()) throw std::invalid_argument("shuffle gadget: lengths differ");
    size_t k = x.size();
    if (k == 1) { cs.constrain(y[0] - LinearCombination(x[0])); return R1CSError::Ok; }
    return cs.specify_randomized_constraints([x, y, k](ConstraintSystem &cs2) {
        Scalar z = cs2.challenge_scalar("shuffle challenge");
        LinearCombination zc(z);
        auto chain = [&](const std::vector<Variable> &v) {
            Variable prev = cs2.multiply(v[k - 1] - zc, v[k - 2] - zc).out;
            for (size_t i = k - 2; i-- > 0;) prev = cs2.multiply(LinearCombination(prev), v[i] - zc).out;
            return prev;
        };
        Variable ox = chain(x), oy = chain(y);
        cs2.constrain(ox - LinearCombination(oy));
        return R1CSError::Ok;
    });
}
void example_gadget(ConstraintSystem &cs, LinearCombination a1, LinearCombination a2, LinearCombination b1, LinearCombination b2, LinearCombination c1, LinearCombination c2) {
    Variable c_var = cs.multiply(a1 + a2, b1 + b2).out;
    cs.constrain(c1 + c2 - LinearCombination(c_var));
}
R1CSError range_proof_gadget(ConstraintSystem &cs, LinearCombination v, const uint64_t *v_assignment, size_t n) {
    Scalar exp_2 = Scalar::one();
    for (size_t i = 0; i < n; i++) {
        std::pair<Scalar, Scalar> asg; const std::pair<Scalar, Scalar> *pa = nullptr;
        if (v_assignment) { uint64_t bit = (*v_assignment >> i) & 1; asg = {Scalar::from_u64(1 - bit), Scalar::from_u64(bit)}; pa = &asg; }
        Multiplier mv; R1CSError e = cs.allocate_multiplier(pa, mv); if (e != R1CSError::Ok) return e;
        cs.constrain(LinearCombination(mv.out));
        cs.constrain(mv.left + (mv.right - LinearCombination(Scalar::one())));
        v = v - mv.right * exp_2;
        exp_2 = exp_2 + exp_2;
    }
    cs.constrain(v);
    return R1CSError::Ok;
}

}  // namespace r1cs
}  // namespace bulletproofs

// ================================================================================================ C shim for the Python harness
using namespace bulletproofs;
using namespace bulletproofs::r1cs;
static R1CSError build_gadget(ConstraintSystem &cs, int gadget, const std::vector<Variable> &vars, uint64_t param, const uint64_t *aux) {
    size_t m = vars.size();
    if (gadget == 0) { if (m < 2 || m % 2) return R1CSError::FormatError; return shuffle_gadget(cs, std::vector<Variable>(vars.begin(), vars.begin() + m / 2), std::vector<Variable>(vars.begin() + m / 2, vars.end())); }
    if (gadget == 1) { if (m != 5) return R1CSError::FormatError; example_gadget(cs, vars[0], vars[1], vars[2], vars[3], vars[4], LinearCombination(Scalar::from_u64(param))); return R1CSError::Ok; }
    if (gadget == 2) { if (m != 1 || param > 64) return R1CSError::FormatError; return range_proof_gadget(cs, vars[0], aux, (size_t)param); }
    return R1CSError::FormatError;
}
extern "C" {
int bph_r1cs_prove(bp_ctx *ctx, bp_gens *gens, size_t gens_capacity, size_t party_capacity, uint8_t *transcript, int gadget, const uint8_t *values, const uint8_t *blindings, size_t m,
                   uint64_t param, uint64_t aux, const uint8_t ext_seed[32], uint8_t *proof_out, size_t *proof_len, uint8_t *commitments_out) {
    try {
        Device dev(ctx); BulletproofGens g{gens, gens_capacity, party_capacity}; Transcript t(transcript); ChaChaRng ext(ext_seed);
        Prover prover(dev, g, t);
        std::vector<Variable> vars; std::vector<Scalar> vs(m), bs(m);
        for (size_t i = 0; i < m; i++) if (!Scalar::from_canonical_bytes(values + 32 * i, vs[i]) || !Scalar::from_canonical_bytes(blindings + 32 * i, bs[i])) return -3;
        auto cvs = prover.commit_vec(vs, bs);
        for (size_t i = 0; i < m; i++) { memcpy(commitments_out + 32 * i, cvs[i].first.data(), 32); vars.push_back(cvs[i].second); }
        R1CSError e = build_gadget(prover, gadget, vars, param, &aux); if (e != R1CSError::Ok) return (int)e;
        R1CSProof proof; e = prover.prove(ext, proof); if (e != R1CSError::Ok) return (int)e;
        std::vector<uint8_t> bytes = proof.to_bytes(); memcpy(proof_out, bytes.data(), bytes.size()); *proof_len = bytes.size();
        t.to_wire(transcript);
        return 0;
    } catch (const std::exception &) { return -1; }
}
int bph_r1cs_verify(bp_ctx *ctx, bp_gens *gens, size_t gens_capacity, size_t party_capacity, const uint8_t *transcript, int gadget, const uint8_t *commitments, size_t m,
                    uint64_t param, const uint8_t *proof, size_t proof_len, const uint8_t ext_seed[32]) {
    try {
        Device dev(ctx); BulletproofGens g{gens, gens_capacity, party_capacity}; Transcript t(transcript); ChaChaRng ext(ext_seed);
        R1CSProof p; R1CSError e = R1CSProof::from_bytes(proof, proof_len, p); if (e != R1CSError::Ok) return (int)e;
        Verifier verifier(dev, g, t);
        std::vector<Variable> vars;
        for (size_t i = 0; i < m; i++) { CompressedRistretto V; memcpy(V.data(), commitments + 32 * i, 32); vars.push_back(verifier.commit(V)); }
        e = build_gadget(verifier, gadget, vars, param, nullptr); if (e != R1CSError::Ok) return (int)e;
        return (int)verifier.verify(p, ext);
    } catch (const std::exception &) { return -1; }
}
}
