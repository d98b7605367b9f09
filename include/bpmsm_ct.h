/* bpmsm_ct.h -- the engine's constant-time entry points, for secret scalars (prover side).
 *
 * Same library (libbpmsm.so), wire types, ownership and threading rules as include/bpmsm.h.  Kept in a header of its own because
 * these calls carry a different contract: their control flow, launches, grids, memory addresses and copies are a function of the
 * public arguments only (term counts, offsets, point indices), never of the scalars; see the "Timing" paragraph of bpmsm.h and
 * DESIGN.md "constant-time policy".  Python binds them in bulletproofs_b200.CT_SYMBOLS.
 */
#ifndef BPMSM_CT_H
#define BPMSM_CT_H
#include "bpmsm.h"
#ifdef __cplusplus
extern "C" {
#endif

/* Indexed MSM over generator-table slots, constant-time in the scalars: the reference's constant-time RistrettoPoint::multiscalar_mul over
 * generators -- PedersenGens::commit (generators.rs:40; V, T_1, T_2 of party.rs:51,216-217, the R1CS commit and T_1, T_3..T_6 of
 * r1cs/prover.rs:284,587-591), A and S (party.rs:100-124), the R1CS A_I, A_O, S (r1cs/prover.rs:433-516).  point_idx[t] must be a table
 * slot of `gens` (no dynamic points).  Same argument checks and status codes as bp_msm_indexed_batch: BP_ERR_INVALID_ARGUMENT for a bad
 * slot, a NULL gens or n_msm = 0, BP_ERR_LENGTH_MISMATCH for decreasing offsets, status[j] = BP_ERR_NONCANONICAL_SCALAR for an MSM
 * holding a scalar >= l.  The device copy of the scalars is zeroed on the context's stream before the call returns. */
int bp_msm_indexed_batch_ct(bp_ctx *ctx, bp_gens *gens, const uint8_t *scalars, const uint32_t *point_idx, const uint64_t *offsets,
                            size_t n_msm, uint8_t *outs, uint8_t *status);

#ifdef __cplusplus
}
#endif
#endif
