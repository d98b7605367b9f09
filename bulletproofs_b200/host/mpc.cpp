// Host mirror of the aggregated range-proof MPC protocol (see mpc.hpp).  Point arithmetic: libbpmsm.so only.
#include "mpc.hpp"

namespace bulletproofs {
namespace mpc {

static void check(int rc, bp_ctx *ctx, const char *what) {
    if (rc == BP_OK) return;
    throw std::runtime_error(std::string(what) + " failed with code " + std::to_string(rc) + ": " + bp_last_error(ctx));
}
static std::vector<uint8_t> pack(const std::vector<Scalar> &v) { std::vector<uint8_t> o(32 * v.size()); for (size_t i = 0; i < v.size(); i++) v[i].write(o.data() + 32 * i); return o; }
static bool valid_bitsize(size_t n) { return n == 8 || n == 16 || n == 32 || n == 64; }
static bool is_identity(const uint8_t p[32]) { uint8_t z = 0; for (int i = 0; i < 32; i++) z |= p[i]; return z == 0; }
static Scalar sum_of_powers(const Scalar &x, size_t n) {            // util.rs:240-262 (n is a power of two or small; the slow form is always right)
    Scalar acc = Scalar::zero(), e = Scalar::one();
    for (size_t i = 0; i < n; i++) { acc += e; e *= x; }
    return acc;
}
// sum of compressed points: one MSM with unit scalars per list (dealer.rs:112-116,169-170); all lists have the same length
static void sum_points(Device &dev, const std::vector<std::vector<CompressedRistretto>> &lists, std::vector<CompressedRistretto> &sums) {
    size_t k = lists.size(), m = lists[0].size();
    std::vector<uint8_t> sc(32 * k * m), pts(32 * k * m), outs(32 * k), st(k); std::vector<uint64_t> offs(k + 1);
    Bytes32 one = Scalar::one().to_bytes();
    for (size_t a = 0; a < k; a++) { offs[a] = a * m; for (size_t j = 0; j < m; j++) { memcpy(sc.data() + 32 * (a * m + j), one.data(), 32); memcpy(pts.data() + 32 * (a * m + j), lists[a][j].data(), 32); } }
    offs[k] = k * m;
    check(bp_msm_batch(dev.ctx, sc.data(), pts.data(), offs.data(), k, outs.data(), st.data()), dev.ctx, "bp_msm_batch");
    sums.resize(k);
    for (size_t a = 0; a < k; a++) { if (st[a] != BP_OK) throw std::invalid_argument("MPC message holds an invalid point encoding"); memcpy(sums[a].data(), outs.data() + 32 * a, 32); }
}

// ------------------------------------------------------------------ messages
bool ProofShare::check_size(size_t expected_n, const BulletproofGens &gens, size_t j) const {
    if (l_vec.size() != expected_n || r_vec.size() != expected_n) return false;
    if (expected_n > gens.gens_capacity) return false;
    if (j >= gens.party_capacity) return false;
    return true;
}
bool ProofShare::audit_share(Device &dev, const BulletproofGens &gens, size_t j, const BitCommitment &bit_commitment, const BitChallenge &bit_challenge,
                             const PolyCommitment &poly_commitment, const PolyChallenge &poly_challenge) const {
    size_t n = l_vec.size();
    if (!check_size(n, gens, j)) return false;
    const Scalar &y = bit_challenge.y, &z = bit_challenge.z, &x = poly_challenge.x;
    Scalar zz = z * z, minus_z = -z, z_j = scalar_exp_vartime(z, (uint64_t)j), y_jn = scalar_exp_vartime(y, (uint64_t)(j * n));
    Scalar y_jn_inv = y_jn.invert(), y_inv = y.invert();
    if (!((t_x - inner_product(l_vec, r_vec)).is_zero())) return false;                                    // :112-114
    // P_check over [A_j, S_j, B~, G_j, H_j] and t_check over [V_j, T_1_j, T_2_j, B, B~] in one device call
    std::vector<Scalar> sc; std::vector<uint32_t> idx; const uint32_t DYN = 0x80000000u;
    sc.push_back(Scalar::one()); idx.push_back(DYN | 0); sc.push_back(x); idx.push_back(DYN | 1); sc.push_back(-e_blinding); idx.push_back(gens.slot_B_blinding());
    for (size_t i = 0; i < n; i++) { sc.push_back(minus_z - l_vec[i]); idx.push_back(gens.slot_G(j, i)); }                     // g :116
    Scalar exp_2 = Scalar::one(), exp_y_inv = Scalar::one(), zzzj = zz * z_j;
    for (size_t i = 0; i < n; i++) {                                                                                            // h :117-125
        Scalar f = exp_y_inv * y_jn_inv;
        sc.push_back(z + f * (-r_vec[i]) + f * (zzzj * exp_2)); idx.push_back(gens.slot_H(j, i));
        exp_2 = exp_2 + exp_2; exp_y_inv *= y_inv;
    }
    size_t split = sc.size();
    Scalar delta = (z - zz) * sum_of_powers(y, n) * y_jn - z * zz * sum_of_powers(Scalar::from_u64(2), n) * z_j;               // :148
    sc.push_back(zzzj); idx.push_back(DYN | 2); sc.push_back(x); idx.push_back(DYN | 3); sc.push_back(x * x); idx.push_back(DYN | 4);
    sc.push_back(delta - t_x); idx.push_back(gens.slot_B()); sc.push_back(-t_x_blinding); idx.push_back(gens.slot_B_blinding());
    uint8_t dyn[5 * 32];
    memcpy(dyn, bit_commitment.A_j.data(), 32); memcpy(dyn + 32, bit_commitment.S_j.data(), 32); memcpy(dyn + 64, bit_commitment.V_j.data(), 32);
    memcpy(dyn + 96, poly_commitment.T_1_j.data(), 32); memcpy(dyn + 128, poly_commitment.T_2_j.data(), 32);
    uint64_t offs[3] = {0, split, sc.size()}; uint8_t outs[64], st[2];
    check(bp_msm_indexed_batch(dev.ctx, gens.handle, pack(sc).data(), idx.data(), dyn, 5, offs, 2, outs, st), dev.ctx, "bp_msm_indexed_batch");
    if (st[0] != BP_OK || st[1] != BP_OK) return false;                                                    // V_j.decompress() -> None :144 (and undecodable A_j, S_j, T_j)
    return is_identity(outs) && is_identity(outs + 32);                                                    // :140-142, :162-166
}
std::vector<uint8_t> ProofShare::to_bytes() const {
    std::vector<uint8_t> o(32 * (3 + l_vec.size() + r_vec.size()));
    t_x.write(o.data()); t_x_blinding.write(o.data() + 32); e_blinding.write(o.data() + 64);
    for (size_t i = 0; i < l_vec.size(); i++) l_vec[i].write(o.data() + 96 + 32 * i);
    for (size_t i = 0; i < r_vec.size(); i++) r_vec[i].write(o.data() + 96 + 32 * (l_vec.size() + i));
    return o;
}
bool ProofShare::from_bytes(const uint8_t *s, size_t n, ProofShare &out) {
    out.l_vec.resize(n); out.r_vec.resize(n);
    bool ok = Scalar::from_canonical_bytes(s, out.t_x) && Scalar::from_canonical_bytes(s + 32, out.t_x_blinding) && Scalar::from_canonical_bytes(s + 64, out.e_blinding);
    for (size_t i = 0; i < n && ok; i++) ok = Scalar::from_canonical_bytes(s + 96 + 32 * i, out.l_vec[i]) && Scalar::from_canonical_bytes(s + 96 + 32 * (n + i), out.r_vec[i]);
    return ok;
}

// ------------------------------------------------------------------ party
MPCError Party::new_(Device &dev, const BulletproofGens &gens, uint64_t v, const Scalar &v_blinding, size_t n, PartyAwaitingPosition &out) {
    if (!valid_bitsize(n)) return MPCError::InvalidBitsize;
    if (gens.gens_capacity < n) return MPCError::InvalidGeneratorsLength;
    std::vector<Scalar> sc = {Scalar::from_u64(v), v_blinding}; uint32_t idx[2] = {gens.slot_B(), gens.slot_B_blinding()}; uint64_t offs[2] = {0, 2}; uint8_t st;
    out = PartyAwaitingPosition{&dev, &gens, n, v, v_blinding, {}};
    check(secret_indexed_msm(dev.ctx, gens.handle, pack(sc).data(), idx, offs, 1, out.V.data(), &st), dev.ctx, "secret_indexed_msm");     // pc_gens.commit :50
    return MPCError::Ok;
}
MPCError PartyAwaitingPosition::assign_position_with_rng(size_t j, Rng &rng, PartyAwaitingBitChallenge &next, BitCommitment &out) const {
    if (gens->party_capacity <= j) return MPCError::InvalidGeneratorsLength;                               // :93-95
    next = PartyAwaitingBitChallenge{dev, gens, n, v, v_blinding, j, Scalar::random(rng), Scalar(), {}, {}};           // a_blinding :98
    next.s_blinding = Scalar::random(rng);                                                                  // :114
    next.s_L.resize(n); next.s_R.resize(n);
    for (size_t i = 0; i < n; i++) next.s_L[i] = Scalar::random(rng);                                       // :115
    for (size_t i = 0; i < n; i++) next.s_R[i] = Scalar::random(rng);                                       // :116
    // A_j = a~ B~ + sum_i (bit ? G_i : -H_i)  (:100-112), written as a~ B~ + sum_i (b_i G_i + (b_i - 1) H_i) so that the point indices do
    // not depend on the bits;  S_j = s~ B~ + <s_L, G> + <s_R, H>  (:119-124): two constant-time MSMs, one call
    std::vector<Scalar> sc; std::vector<uint32_t> idx; Scalar one = Scalar::one();
    sc.push_back(next.a_blinding); idx.push_back(gens->slot_B_blinding());
    for (size_t i = 0; i < n; i++) { Scalar b = Scalar::from_u64((v >> i) & 1); sc.push_back(b); idx.push_back(gens->slot_G(j, i)); sc.push_back(b - one); idx.push_back(gens->slot_H(j, i)); }
    size_t split = sc.size();
    sc.push_back(next.s_blinding); idx.push_back(gens->slot_B_blinding());
    for (size_t i = 0; i < n; i++) { sc.push_back(next.s_L[i]); idx.push_back(gens->slot_G(j, i)); }
    for (size_t i = 0; i < n; i++) { sc.push_back(next.s_R[i]); idx.push_back(gens->slot_H(j, i)); }
    uint64_t offs[3] = {0, split, sc.size()}; uint8_t outs[64], st[2];
    check(secret_indexed_msm(dev->ctx, gens->handle, pack(sc).data(), idx.data(), offs, 2, outs, st), dev->ctx, "secret_indexed_msm");
    out.V_j = V; memcpy(out.A_j.data(), outs, 32); memcpy(out.S_j.data(), outs + 32, 32);
    return MPCError::Ok;
}
void PartyAwaitingBitChallenge::apply_challenge_with_rng(const BitChallenge &vc, Rng &rng, PartyAwaitingPolyChallenge &next, PolyCommitment &out) const {
    const Scalar &y = vc.y, &z = vc.z;
    Scalar one = Scalar::one(), zz = z * z, offset_y = scalar_exp_vartime(y, (uint64_t)(j * n)), offset_z = scalar_exp_vartime(z, (uint64_t)j);
    next = PartyAwaitingPolyChallenge();
    next.offset_zz = zz * offset_z;                                                                         // :199
    next.l0.resize(n); next.l1.resize(n); next.r0.resize(n); next.r1.resize(n);
    Scalar exp_y = offset_y, exp_2 = one;
    for (size_t i = 0; i < n; i++) {                                                                        // :201-211
        Scalar a_L = Scalar::from_u64((v >> i) & 1), a_R = a_L - one;
        next.l0[i] = a_L - z; next.l1[i] = s_L[i];
        next.r0[i] = exp_y * (a_R + z) + next.offset_zz * exp_2; next.r1[i] = exp_y * s_R[i];
        exp_y *= y; exp_2 = exp_2 + exp_2;
    }
    Scalar acc0 = Scalar::zero(), acc2 = Scalar::zero(), acc1 = Scalar::zero();                            // VecPoly1::inner_product, util.rs:86-100
    for (size_t i = 0; i < n; i++) { acc0 += next.l0[i] * next.r0[i]; acc2 += next.l1[i] * next.r1[i]; acc1 += (next.l0[i] + next.l1[i]) * (next.r0[i] + next.r1[i]); }
    next.t0 = acc0; next.t2 = acc2; next.t1 = acc1 - acc0 - acc2;
    next.t_1_blinding = Scalar::random(rng); next.t_2_blinding = Scalar::random(rng);                       // :214-215
    next.v_blinding = v_blinding; next.a_blinding = a_blinding; next.s_blinding = s_blinding;
    std::vector<Scalar> sc = {next.t1, next.t_1_blinding, next.t2, next.t_2_blinding};                      // T_1_j, T_2_j :216-217
    uint32_t idx[4] = {gens->slot_B(), gens->slot_B_blinding(), gens->slot_B(), gens->slot_B_blinding()}; uint64_t offs[3] = {0, 2, 4}; uint8_t outs[64], st[2];
    check(secret_indexed_msm(dev->ctx, gens->handle, pack(sc).data(), idx, offs, 2, outs, st), dev->ctx, "secret_indexed_msm");
    memcpy(out.T_1_j.data(), outs, 32); memcpy(out.T_2_j.data(), outs + 32, 32);
}
MPCError PartyAwaitingPolyChallenge::apply_challenge(const PolyChallenge &pc, ProofShare &out) const {
    if (pc.x.is_zero()) return MPCError::MaliciousDealer;                                                   // :282-284
    const Scalar &x = pc.x; size_t n = l0.size();
    out.t_x = t0 + x * (t1 + x * t2);                                                                       // :286-294
    out.t_x_blinding = offset_zz * v_blinding + x * (t_1_blinding + x * t_2_blinding);
    out.e_blinding = a_blinding + s_blinding * x;
    out.l_vec.resize(n); out.r_vec.resize(n);
    for (size_t i = 0; i < n; i++) { out.l_vec[i] = l0[i] + l1[i] * x; out.r_vec[i] = r0[i] + r1[i] * x; }
    return MPCError::Ok;
}

// ------------------------------------------------------------------ dealer
MPCError Dealer::new_(Device &dev, const BulletproofGens &gens, Transcript &transcript, size_t n, size_t m, DealerAwaitingBitCommitments &out) {
    if (!valid_bitsize(n)) return MPCError::InvalidBitsize;
    if (m == 0 || (m & (m - 1))) return MPCError::InvalidAggregation;
    if (gens.gens_capacity < n || gens.party_capacity < m) return MPCError::InvalidGeneratorsLength;
    out.dev = &dev; out.gens = &gens; out.n = n; out.m = m; out.transcript = &transcript;
    out.initial_transcript = transcript;                                                                    // cloned before the domain separator (:57-68)
    transcript.rangeproof_domain_sep(n, m);                                                                 // :70
    return MPCError::Ok;
}
MPCError DealerAwaitingBitCommitments::receive_bit_commitments(const std::vector<BitCommitment> &bcs, DealerAwaitingPolyCommitments &next, BitChallenge &out) const {
    if (m != bcs.size()) return MPCError::WrongNumBitCommitments;
    for (const BitCommitment &vc : bcs) transcript->append_point("V", vc.V_j);
    std::vector<std::vector<CompressedRistretto>> lists(2); std::vector<CompressedRistretto> sums;
    for (const BitCommitment &vc : bcs) { lists[0].push_back(vc.A_j); lists[1].push_back(vc.S_j); }
    sum_points(*dev, lists, sums);
    transcript->append_point("A", sums[0]); transcript->append_point("S", sums[1]);
    out.y = transcript->challenge_scalar("y"); out.z = transcript->challenge_scalar("z");
    next.dev = dev; next.gens = gens; next.n = n; next.m = m; next.transcript = transcript; next.initial_transcript = initial_transcript;
    next.bit_challenge = out; next.bit_commitments = bcs; next.A = sums[0]; next.S = sums[1];
    return MPCError::Ok;
}
MPCError DealerAwaitingPolyCommitments::receive_poly_commitments(const std::vector<PolyCommitment> &pcs, DealerAwaitingProofShares &next, PolyChallenge &out) const {
    if (m != pcs.size()) return MPCError::WrongNumPolyCommitments;
    std::vector<std::vector<CompressedRistretto>> lists(2); std::vector<CompressedRistretto> sums;
    for (const PolyCommitment &pc : pcs) { lists[0].push_back(pc.T_1_j); lists[1].push_back(pc.T_2_j); }
    sum_points(*dev, lists, sums);
    transcript->append_point("T_1", sums[0]); transcript->append_point("T_2", sums[1]);
    out.x = transcript->challenge_scalar("x");
    next.dev = dev; next.gens = gens; next.n = n; next.m = m; next.transcript = transcript; next.initial_transcript = initial_transcript;
    next.bit_challenge = bit_challenge; next.bit_commitments = bit_commitments; next.poly_challenge = out; next.poly_commitments = pcs;
    next.A = A; next.S = S; next.T_1 = sums[0]; next.T_2 = sums[1];
    return MPCError::Ok;
}
MPCError DealerAwaitingProofShares::assemble_shares(const std::vector<ProofShare> &shares, RangeProof &proof, std::vector<size_t> &bad_shares) {
    if (m != shares.size()) return MPCError::WrongNumProofShares;
    bad_shares.clear();
    for (size_t j = 0; j < m; j++) if (!shares[j].check_size(n, *gens, j)) bad_shares.push_back(j);
    if (!bad_shares.empty()) return MPCError::MalformedProofShares;
    proof.t_x = Scalar::zero(); proof.t_x_blinding = Scalar::zero(); proof.e_blinding = Scalar::zero();
    for (const ProofShare &ps : shares) { proof.t_x += ps.t_x; proof.t_x_blinding += ps.t_x_blinding; proof.e_blinding += ps.e_blinding; }
    transcript->append_scalar("t_x", proof.t_x); transcript->append_scalar("t_x_blinding", proof.t_x_blinding); transcript->append_scalar("e_blinding", proof.e_blinding);
    Scalar w = transcript->challenge_scalar("w");
    CompressedRistretto Q; uint32_t qi = gens->slot_B(); uint64_t qo[2] = {0, 1}; uint8_t qs;                // Q = w B :256
    check(bp_msm_indexed_batch(dev->ctx, gens->handle, w.to_bytes().data(), &qi, nullptr, 0, qo, 1, Q.data(), &qs), dev->ctx, "bp_msm_indexed_batch");
    size_t N = n * m;
    std::vector<Scalar> Gf(N, Scalar::one()), Hf(N), l_vec, r_vec;
    Scalar y_inv = bit_challenge.y.invert(), e = Scalar::one();
    for (size_t i = 0; i < N; i++) { Hf[i] = e; e *= y_inv; }
    for (const ProofShare &ps : shares) { l_vec.insert(l_vec.end(), ps.l_vec.begin(), ps.l_vec.end()); r_vec.insert(r_vec.end(), ps.r_vec.begin(), ps.r_vec.end()); }
    proof.ipp_proof = InnerProductProof::create(*dev, *gens, n, m, *transcript, Q, Gf, Hf, std::move(l_vec), std::move(r_vec));
    proof.A = A; proof.S = S; proof.T_1 = T_1; proof.T_2 = T_2;
    return MPCError::Ok;
}
MPCError DealerAwaitingProofShares::receive_shares(const std::vector<ProofShare> &shares, RangeProof &proof, std::vector<size_t> &bad_shares) {
    MPCError e = assemble_shares(shares, proof, bad_shares);
    if (e != MPCError::Ok) return e;
    std::vector<CompressedRistretto> Vs; for (const BitCommitment &vc : bit_commitments) Vs.push_back(vc.V_j);
    if (proof.verify_multiple(*dev, *gens, initial_transcript, Vs, n) == ProofError::Ok) return MPCError::Ok;                       // :330-337
    for (size_t j = 0; j < m; j++)                                                                                                   // :340-353
        if (!shares[j].audit_share(*dev, *gens, j, bit_commitments[j], bit_challenge, poly_commitments[j], poly_challenge)) bad_shares.push_back(j);
    return MPCError::MalformedProofShares;
}
MPCError DealerAwaitingProofShares::receive_trusted_shares(const std::vector<ProofShare> &shares, RangeProof &proof) {
    std::vector<size_t> bad; return assemble_shares(shares, proof, bad);
}

}  // namespace mpc
}  // namespace bulletproofs

// ------------------------------------------------------------------ C shim for the Python harness: the stateless form the oracle exposes (oracle/mpc.h) —
// a party is (v, v_blinding, n, j, seed); every stage replays the party's ChaCha stream through the typestate structs above.
using namespace bulletproofs;
using namespace bulletproofs::mpc;
namespace {
struct PartyRun { PartyAwaitingPosition p0; PartyAwaitingBitChallenge p1; PartyAwaitingPolyChallenge p2; BitCommitment bc; PolyCommitment pc; };
MPCError run_party(Device &dev, const BulletproofGens &g, uint64_t v, const uint8_t *v_blinding, size_t n, size_t j, const uint8_t seed[32], const uint8_t *y, const uint8_t *z,
                   PartyRun &r, bool &bad_scalar) {
    Scalar vb; bad_scalar = !Scalar::from_canonical_bytes(v_blinding, vb);
    if (bad_scalar) return MPCError::Ok;
    ChaChaRng rng(seed);
    MPCError e = Party::new_(dev, g, v, vb, n, r.p0); if (e != MPCError::Ok) return e;
    e = r.p0.assign_position_with_rng(j, rng, r.p1, r.bc); if (e != MPCError::Ok) return e;
    if (!y) return MPCError::Ok;
    BitChallenge c; bad_scalar = !Scalar::from_canonical_bytes(y, c.y) || !Scalar::from_canonical_bytes(z, c.z);
    if (bad_scalar) return MPCError::Ok;
    r.p1.apply_challenge_with_rng(c, rng, r.p2, r.pc);
    return MPCError::Ok;
}
}  // namespace
extern "C" {
int bph_mpc_party_bit_commitment(bp_ctx *ctx, bp_gens *gens, size_t gens_capacity, size_t party_capacity, uint64_t v, const uint8_t v_blinding[32], size_t n, size_t j,
                                 const uint8_t seed[32], uint8_t out[96]) {
    try {
        Device dev(ctx); BulletproofGens g{gens, gens_capacity, party_capacity}; PartyRun r; bool bad;
        MPCError e = run_party(dev, g, v, v_blinding, n, j, seed, nullptr, nullptr, r, bad);
        if (bad) return 7;
        if (e != MPCError::Ok) return (int)e;
        memcpy(out, r.bc.V_j.data(), 32); memcpy(out + 32, r.bc.A_j.data(), 32); memcpy(out + 64, r.bc.S_j.data(), 32);
        return 0;
    } catch (const std::exception &) { return -1; }
}
int bph_mpc_party_poly_commitment(bp_ctx *ctx, bp_gens *gens, size_t gens_capacity, size_t party_capacity, uint64_t v, size_t n, size_t j, const uint8_t seed[32],
                                  const uint8_t y[32], const uint8_t z[32], uint8_t out[64]) {
    try {
        Device dev(ctx); BulletproofGens g{gens, gens_capacity, party_capacity}; PartyRun r; bool bad; uint8_t zero[32] = {0};
        MPCError e = run_party(dev, g, v, zero, n, j, seed, y, z, r, bad);         // the blinding of V does not enter T_1_j, T_2_j
        if (bad) return 7;
        if (e != MPCError::Ok) return (int)e;
        memcpy(out, r.pc.T_1_j.data(), 32); memcpy(out + 32, r.pc.T_2_j.data(), 32);
        return 0;
    } catch (const std::exception &) { return -1; }
}
int bph_mpc_party_proof_share(bp_ctx *ctx, bp_gens *gens, size_t gens_capacity, size_t party_capacity, uint64_t v, const uint8_t v_blinding[32], size_t n, size_t j,
                              const uint8_t seed[32], const uint8_t y[32], const uint8_t z[32], const uint8_t x[32], uint8_t *out) {
    try {
        Device dev(ctx); BulletproofGens g{gens, gens_capacity, party_capacity}; PartyRun r; bool bad;
        MPCError e = run_party(dev, g, v, v_blinding, n, j, seed, y, z, r, bad);
        PolyChallenge pc; if (bad || !Scalar::from_canonical_bytes(x, pc.x)) return 7;
        if (e != MPCError::Ok) return (int)e;
        ProofShare sh; e = r.p2.apply_challenge(pc, sh); if (e != MPCError::Ok) return (int)e;
        std::vector<uint8_t> b = sh.to_bytes(); memcpy(out, b.data(), b.size());
        return 0;
    } catch (const std::exception &) { return -1; }
}
int bph_mpc_audit_share(bp_ctx *ctx, bp_gens *gens, size_t gens_capacity, size_t party_capacity, size_t n, size_t j, const uint8_t bitc[96], const uint8_t y[32],
                        const uint8_t z[32], const uint8_t polyc[64], const uint8_t x[32], const uint8_t *share) {
    try {
        Device dev(ctx); BulletproofGens g{gens, gens_capacity, party_capacity};
        BitChallenge bch; PolyChallenge pch;
        if (!Scalar::from_canonical_bytes(y, bch.y) || !Scalar::from_canonical_bytes(z, bch.z) || !Scalar::from_canonical_bytes(x, pch.x)) return 7;
        ProofShare sh; if (!ProofShare::from_bytes(share, n, sh)) return 1;
        BitCommitment bc; memcpy(bc.V_j.data(), bitc, 32); memcpy(bc.A_j.data(), bitc + 32, 32); memcpy(bc.S_j.data(), bitc + 64, 32);
        PolyCommitment pc; memcpy(pc.T_1_j.data(), polyc, 32); memcpy(pc.T_2_j.data(), polyc + 32, 32);
        return sh.audit_share(dev, g, j, bc, bch, pc, pch) ? 0 : 1;
    } catch (const std::exception &) { return -1; }
}
// The whole dealer over collected messages (Dealer::new .. receive_shares / receive_trusted_shares); transcript: 203-byte wire state, in = initial, out = final.
// challenges_out = y | z | x (96 B, may be null); bad[j] = 1 for every share reported in MalformedProofShares.
int bph_mpc_dealer_run(bp_ctx *ctx, bp_gens *gens, size_t gens_capacity, size_t party_capacity, uint8_t *transcript, size_t n, size_t m, const uint8_t *bitc,
                       const uint8_t *polyc, const uint8_t *shares, int trusted, uint8_t *proof_out, uint8_t *bad, uint8_t *challenges_out) {
    try {
        Device dev(ctx); BulletproofGens g{gens, gens_capacity, party_capacity}; Transcript t(transcript);
        DealerAwaitingBitCommitments d0; DealerAwaitingPolyCommitments d1; DealerAwaitingProofShares d2;
        MPCError e = Dealer::new_(dev, g, t, n, m, d0); if (e != MPCError::Ok) return (int)e;
        std::vector<BitCommitment> bcs(m); std::vector<PolyCommitment> pcs(m); std::vector<ProofShare> shs(m);
        for (size_t j = 0; j < m; j++) { memcpy(bcs[j].V_j.data(), bitc + 96 * j, 32); memcpy(bcs[j].A_j.data(), bitc + 96 * j + 32, 32); memcpy(bcs[j].S_j.data(), bitc + 96 * j + 64, 32); }
        BitChallenge bch; e = d0.receive_bit_commitments(bcs, d1, bch); if (e != MPCError::Ok) return (int)e;
        if (challenges_out) { bch.y.write(challenges_out); bch.z.write(challenges_out + 32); }
        if (!polyc) { t.to_wire(transcript); return 0; }
        for (size_t j = 0; j < m; j++) { memcpy(pcs[j].T_1_j.data(), polyc + 64 * j, 32); memcpy(pcs[j].T_2_j.data(), polyc + 64 * j + 32, 32); }
        PolyChallenge pch; e = d1.receive_poly_commitments(pcs, d2, pch); if (e != MPCError::Ok) return (int)e;
        if (challenges_out) pch.x.write(challenges_out + 64);
        if (!shares) { t.to_wire(transcript); return 0; }
        memset(bad, 0, m);
        size_t slen = 32 * (3 + 2 * n); bool malformed = false;
        for (size_t j = 0; j < m; j++) if (!ProofShare::from_bytes(shares + slen * j, n, shs[j])) { bad[j] = 1; malformed = true; }
        if (malformed) return (int)MPCError::MalformedProofShares;
        RangeProof proof; std::vector<size_t> bad_shares;
        e = trusted ? d2.receive_trusted_shares(shs, proof) : d2.receive_shares(shs, proof, bad_shares);
        for (size_t j : bad_shares) bad[j] = 1;
        if (e != MPCError::Ok) return (int)e;
        std::vector<uint8_t> bytes = proof.to_bytes(); memcpy(proof_out, bytes.data(), bytes.size());
        t.to_wire(transcript);
        return 0;
    } catch (const std::invalid_argument &) { return 6; } catch (const std::exception &) { return -1; }
}
}  // extern "C"
