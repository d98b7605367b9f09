"""GPU tier of the constant-time indexed MSM (bp_msm_indexed_batch_ct): results against the oracle and against the variable-time
bp_msm_indexed_batch, edge scalars, the error contract, and a launch sequence that does not depend on the scalars."""
import ctypes
import json
import os
import random

import pytest

from oracle_binding import L_ORDER as l

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EDGE = [0, 1, 8, 15, 16, l - 1, 2**252, int("08" * 31 + "88", 16), int("0" + "7" * 62 + "8", 16), int("8" * 63, 16) % l, 2**128 - 1, l - 2**200]
CAP = 1 << 14


def le(x):
    return x.to_bytes(32, "little")


@pytest.fixture(scope="module")
def G(gpu_ctx):
    import bulletproofs_b200 as bp
    g = bp.Gens(gpu_ctx, CAP, 1)
    yield g
    g.close()


@pytest.fixture(scope="module")
def table(G):
    """compressed point of every slot used below (B~, B, G[0][i], H[0][i])"""
    return [G.B_blinding, G.B] + [G.G(0, i) for i in range(CAP)] + [G.H(0, i) for i in range(CAP)]


def check(G, orc, table, scalars, idx, offsets, with_vartime=True):
    sc = b"".join(le(x) for x in scalars)
    st, got = G.msm_indexed(sc, idx, offsets, constant_time=True)
    assert st == [0] * (len(offsets) - 1)
    if with_vartime:
        st2, want = G.msm_indexed(sc, idx, offsets)
        assert st2 == st and got == want
    for j in range(len(offsets) - 1):
        a, b = offsets[j], offsets[j + 1]
        if a == b:
            assert got[j] == bytes(32); continue
        rc, o = orc.msm(sc[32 * a:32 * b], b"".join(table[i] for i in idx[a:b]))
        assert rc == 0 and got[j] == o, (j, b - a)
    return got


@pytest.mark.parametrize("n", [1, 2, 3, 129, 2064])
def test_single_msm_matches_oracle_and_vartime(G, orc, table, n):
    rnd = random.Random(31 + n)
    idx = [rnd.randrange(len(table)) for _ in range(n)]
    check(G, orc, table, [rnd.randrange(l) for _ in range(n)], idx, [0, n])


def test_prover_shapes(G, orc, table):
    """1024 Pedersen commitments (2 terms each) in one call; the S of a (64, 16) proof of prove_many, 16 x 129 terms in one MSM"""
    rnd = random.Random(32)
    idx = [1, 0] * 1024
    check(G, orc, table, [rnd.randrange(l) for _ in range(2048)], idx, list(range(0, 2049, 2)))
    idx = []
    for j in range(16):
        idx += [0] + [G.slot_G(0, 64 * j + i) for i in range(64)] + [G.slot_H(0, 64 * j + i) for i in range(64)]
    check(G, orc, table, [rnd.randrange(l) for _ in range(len(idx))], idx, [0, len(idx)])


def test_ragged_offsets_and_edge_scalars(G, orc, table):
    rnd = random.Random(33)
    lens = [1, 0, 2, 3, 0, 17, len(EDGE), 64, 5, 129, 1, 300, 33]
    offsets = [0]
    for n in lens:
        offsets.append(offsets[-1] + n)
    T = offsets[-1]
    scalars = [rnd.randrange(l) for _ in range(T)]
    e0 = offsets[lens.index(len(EDGE))]
    scalars[e0:e0 + len(EDGE)] = EDGE
    idx = [rnd.randrange(len(table)) for _ in range(T)]
    idx[offsets[3]:offsets[4]] = [5, 5, 5]                  # repeated slot in one MSM
    check(G, orc, table, scalars, idx, offsets)
    # every edge scalar alone, and all-zero scalars (result: the identity, 32 zero bytes)
    check(G, orc, table, EDGE, [7] * len(EDGE), list(range(len(EDGE) + 1)))
    st, got = G.msm_indexed(bytes(32 * 40), list(range(40)), [0, 40], constant_time=True)
    assert st == [0] and got == [bytes(32)]


def test_large_msm(G, orc, table):
    n = (1 << 15) + 1
    rnd = random.Random(34)
    check(G, orc, table, [rnd.randrange(l) for _ in range(n)], [rnd.randrange(len(table)) for _ in range(n)], [0, n], with_vartime=False)


def test_errors(gpu_ctx, G, golden):
    import bulletproofs_b200 as bp
    rnd = random.Random(35)
    sc = [le(rnd.randrange(l)) for _ in range(6)]
    bad = sc[:4] + [le(l)] + sc[5:]
    st, _ = G.msm_indexed(b"".join(bad), [1, 0, 2, 3, 4, 5], [0, 3, 6], constant_time=True)
    assert st == [0, bp.ERR_NONCANONICAL_SCALAR]          # only the MSM holding the scalar >= l
    L = bp.ct_lib()
    idx, outs, status = (ctypes.c_uint32 * 2)(1, 0), ctypes.create_string_buffer(64), ctypes.create_string_buffer(2)
    s2 = b"".join(sc[:2])
    def call(gens_h, idx_, offs, n_msm):
        return L.bp_msm_indexed_batch_ct(gpu_ctx._h, gens_h, s2, idx_, (ctypes.c_uint64 * len(offs))(*offs), n_msm, outs, status)
    assert call(G._h, (ctypes.c_uint32 * 2)(1, 2 + 2 * CAP), [0, 2], 1) == bp.ERR_INVALID_ARGUMENT              # slot past the table
    assert call(G._h, (ctypes.c_uint32 * 2)(1, 0x80000000), [0, 2], 1) == bp.ERR_INVALID_ARGUMENT              # dynamic point
    assert call(None, idx, [0, 2], 1) == bp.ERR_INVALID_ARGUMENT
    assert call(G._h, idx, [0, 2], 0) == bp.ERR_INVALID_ARGUMENT
    assert call(G._h, idx, [0, 2, 1, 2], 3) == bp.ERR_LENGTH_MISMATCH
    # a pending verification owns the context's scratch
    proof = bytes.fromhex([p for p in golden["proofs"] if p["n"] == 64 and p["m"] == 1][0]["proof"])
    vc = bytes.fromhex(golden["value_commitments"][0])
    g64 = bp.Gens(gpu_ctx, 64, 1)
    try:
        t = bp.Transcript(golden["transcript_label"].encode())
        assert L.bp_rangeproof_verify_begin(gpu_ctx._h, g64._h, t.to_bytes(), proof, len(proof), vc, 64, 1, 1, bytes(32)) == 0
        assert call(G._h, idx, [0, 2], 1) == bp.ERR_INVALID_ARGUMENT
        v = ctypes.create_string_buffer(1)
        assert L.bp_rangeproof_verify_finish(gpu_ctx._h, v) == 0 and v.raw == b"\x00"
    finally:
        g64.close()
    assert call(G._h, idx, [0, 2], 1) == 0


def test_launch_sequence_does_not_depend_on_the_scalars(gpu_ctx, G):
    """per-kernel launch counts (event profiler) and the launch total for all-zero, all-(l-1) and random scalars of one shape"""
    rnd = random.Random(36)
    offsets = [0, 1, 3, 3, 70, 200, 201]
    T = offsets[-1]
    idx = [rnd.randrange(2 + 2 * CAP) for _ in range(T)]
    seen = []
    for scalars in ([0] * T, [l - 1] * T, [rnd.randrange(l) for _ in range(T)]):
        gpu_ctx.prof_enable(True)
        n0 = gpu_ctx.launches
        G.msm_indexed(b"".join(le(x) for x in scalars), idx, offsets, constant_time=True)
        counts = {k: v[1] for k, v in gpu_ctx.prof_report().items()}
        seen.append((counts, gpu_ctx.launches - n0))
        gpu_ctx.prof_enable(False)
    assert seen[0] == seen[1] == seen[2], seen
    assert {"k_msm_ct_recode", "k_msm_ct_table", "k_msm_ct_straus", "k_msm_ct_reduce"} <= set(seen[0][0])
