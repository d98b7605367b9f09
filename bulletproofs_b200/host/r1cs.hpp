// C++ mirror of the reference's r1cs module (feature `yoloproofs`) above the C ABI:
//   Variable, LinearCombination            /root/reference/src/r1cs/linear_combination.rs
//   ConstraintSystem traits                /root/reference/src/r1cs/constraint_system.rs
//   Prover::{new, commit, prove}           /root/reference/src/r1cs/prover.rs:242-698
//   Verifier::{new, commit, verify}        /root/reference/src/r1cs/verifier.rs:204-500
//   R1CSProof::{to_bytes, from_bytes}      /root/reference/src/r1cs/proof.rs:71-204
// Every multiscalar multiplication runs on the GPU: the commitments to secrets (commit, A_I/A_O/S in both phases, the
// T commitments) through the constant-time bp_msm_indexed_batch_ct; Q, the IPP rounds and the verifier's mega-check through
// the variable-time bp_msm_indexed_batch / bp_ippx_*, as the reference does.
#pragma once
#include <functional>
#include <memory>
#include "bulletproofs.hpp"

namespace bulletproofs {
namespace r1cs {

enum class VarKind { Committed, MultiplierLeft, MultiplierRight, MultiplierOutput, One };
struct Variable { VarKind kind; size_t index; static Variable One() { return {VarKind::One, 0}; } };

struct LinearCombination {
    std::vector<std::pair<Variable, Scalar>> terms;
    LinearCombination() {}
    LinearCombination(Variable v) { terms.push_back({v, Scalar::one()}); }                 // From<Variable>
    LinearCombination(const Scalar &s) { terms.push_back({Variable::One(), s}); }          // From<Scalar>
    LinearCombination operator+(const LinearCombination &o) const { LinearCombination r = *this; r.terms.insert(r.terms.end(), o.terms.begin(), o.terms.end()); return r; }
    LinearCombination operator-(const LinearCombination &o) const { LinearCombination r = *this; for (auto &t : o.terms) r.terms.push_back({t.first, -t.second}); return r; }
    LinearCombination operator*(const Scalar &s) const { LinearCombination r = *this; for (auto &t : r.terms) t.second = t.second * s; return r; }
    LinearCombination operator-() const { LinearCombination r = *this; for (auto &t : r.terms) t.second = -t.second; return r; }
};
inline LinearCombination operator-(Variable a, const LinearCombination &b) { return LinearCombination(a) - b; }
inline LinearCombination operator+(Variable a, const LinearCombination &b) { return LinearCombination(a) + b; }
inline LinearCombination operator*(Variable a, const Scalar &s) { LinearCombination r; r.terms.push_back({a, s}); return r; }

enum class R1CSError { Ok = 0, VerificationError = 1, FormatError = 2, InvalidGeneratorsLength = 4, MissingAssignment = 9, GadgetError = 10 };

struct Multiplier { Variable left, right, out; };

class ConstraintSystem {                                    // constraint_system.rs:20-91
public:
    virtual ~ConstraintSystem() {}
    virtual Transcript &transcript() = 0;
    virtual Multiplier multiply(LinearCombination left, LinearCombination right) = 0;
    virtual R1CSError allocate(const Scalar *assignment, Variable &out) = 0;
    virtual R1CSError allocate_multiplier(const std::pair<Scalar, Scalar> *assignments, Multiplier &out) = 0;
    virtual size_t multipliers_len() const = 0;
    virtual void constrain(LinearCombination lc) = 0;
    // RandomizableConstraintSystem / RandomizedConstraintSystem (constraint_system.rs:100-135)
    using Callback = std::function<R1CSError(ConstraintSystem &)>;
    virtual R1CSError specify_randomized_constraints(Callback cb) = 0;
    virtual Scalar challenge_scalar(const char *label) = 0;          // only valid inside a randomized callback
};

struct R1CSProof {
    CompressedRistretto A_I1, A_O1, S1, A_I2, A_O2, S2, T_1, T_3, T_4, T_5, T_6;
    Scalar t_x, t_x_blinding, e_blinding; InnerProductProof ipp_proof;
    std::vector<uint8_t> to_bytes() const;
    static R1CSError from_bytes(const uint8_t *s, size_t len, R1CSProof &out);
};

// merlin::TranscriptRng (build_rng / rekey_with_witness_bytes / finalize)
class TranscriptRng : public Rng {
    alignas(8) uint8_t st_[200]; merlin_t m_;
public:
    explicit TranscriptRng(const Transcript &t);
    void rekey_with_witness_bytes(const char *label, const uint8_t *w, size_t len);
    void finalize(Rng &external);
    void fill_bytes(uint8_t *out, size_t n) override;
};

class Prover : public ConstraintSystem {
    Transcript &t_; const BulletproofGens &gens_; Device &dev_;
    std::vector<LinearCombination> constraints_;
    std::vector<Scalar> a_L_, a_R_, a_O_, v_, v_blinding_;
    std::vector<Callback> deferred_; bool pending_ = false; size_t pending_idx_ = 0; bool in_phase2_ = false;
    Scalar eval(const LinearCombination &lc) const;
public:
    Prover(Device &dev, const BulletproofGens &gens, Transcript &t);                         // prover.rs:242-258 (pc_gens = the table's B, B~)
    std::pair<CompressedRistretto, Variable> commit(const Scalar &v, const Scalar &v_blinding);   // prover.rs:278-288
    // the same as calling commit() for each pair in order (identical transcript and commitments), but all Pedersen
    // commitments are computed by one batched GPU call instead of one launch sequence per variable
    std::vector<std::pair<CompressedRistretto, Variable>> commit_vec(const std::vector<Scalar> &v, const std::vector<Scalar> &v_blinding);
    R1CSError prove(Rng &external_rng, R1CSProof &out);                                      // prover.rs:380-698
    Transcript &transcript() override { return t_; }
    Multiplier multiply(LinearCombination left, LinearCombination right) override;
    R1CSError allocate(const Scalar *assignment, Variable &out) override;
    R1CSError allocate_multiplier(const std::pair<Scalar, Scalar> *a, Multiplier &out) override;
    size_t multipliers_len() const override { return a_L_.size(); }
    void constrain(LinearCombination lc) override { constraints_.push_back(std::move(lc)); }
    R1CSError specify_randomized_constraints(Callback cb) override { deferred_.push_back(std::move(cb)); return R1CSError::Ok; }
    Scalar challenge_scalar(const char *label) override { return t_.challenge_scalar(label); }
};

class Verifier : public ConstraintSystem {
    Transcript &t_; const BulletproofGens &gens_; Device &dev_;
    std::vector<LinearCombination> constraints_; std::vector<CompressedRistretto> V_;
    size_t num_vars_ = 0; std::vector<Callback> deferred_; bool pending_ = false; size_t pending_idx_ = 0;
public:
    Verifier(Device &dev, const BulletproofGens &gens, Transcript &t);                       // verifier.rs:204-217
    Variable commit(const CompressedRistretto &V);                                           // verifier.rs:236-245
    R1CSError verify(const R1CSProof &proof, Rng &external_rng);                             // verifier.rs:329-500
    Transcript &transcript() override { return t_; }
    Multiplier multiply(LinearCombination left, LinearCombination right) override;
    R1CSError allocate(const Scalar *assignment, Variable &out) override;
    R1CSError allocate_multiplier(const std::pair<Scalar, Scalar> *a, Multiplier &out) override;
    size_t multipliers_len() const override { return num_vars_; }
    void constrain(LinearCombination lc) override { constraints_.push_back(std::move(lc)); }
    R1CSError specify_randomized_constraints(Callback cb) override { deferred_.push_back(std::move(cb)); return R1CSError::Ok; }
    Scalar challenge_scalar(const char *label) override { return t_.challenge_scalar(label); }
};

// gadgets used by the reference's benches and tests
R1CSError shuffle_gadget(ConstraintSystem &cs, std::vector<Variable> x, std::vector<Variable> y);                      // benches/r1cs.rs:35-67
void example_gadget(ConstraintSystem &cs, LinearCombination a1, LinearCombination a2, LinearCombination b1, LinearCombination b2,
                    LinearCombination c1, LinearCombination c2);                                                        // tests/r1cs.rs:225-236
R1CSError range_proof_gadget(ConstraintSystem &cs, LinearCombination v, const uint64_t *v_assignment, size_t n);        // tests/r1cs.rs:366-385

}  // namespace r1cs
}  // namespace bulletproofs
