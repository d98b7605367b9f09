"""GPU tier: the kernel launches of one call of each C ABI entry point, on fixed seeded inputs.  Per-kernel counts come from the
context's event profiler (Context.prof_report), the total from Context.launches.  A change to the host layer that adds, drops or
moves work between entry points shows up here even when the results stay right."""
import ctypes
import json
import os
import random
from collections import Counter

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PASS = Counter({"k_msm_count": 1, "k_msm_scan": 2, "k_msm_scatter": 1, "k_msm_accumulate": 1, "k_msm_reduce": 1, "k_msm_combine": 1})   # one Pippenger pass
DYN = 0x80000000


def scalars(rnd, n):
    return b"".join(rnd.randbytes(31) + bytes([rnd.randrange(16)]) for _ in range(n))      # < 2^252: canonical


def points(ctx, rnd, n):
    return ctx.from_uniform_bytes(rnd.randbytes(64 * n))


def golden_rangeproof():
    g = json.load(open(os.path.join(ROOT, "tests", "golden", "range_proof_v1.json")))
    proof = bytes.fromhex([p for p in g["proofs"] if p["n"] == 64 and p["m"] == 1][0]["proof"])
    return g["transcript_label"].encode(), proof, bytes.fromhex(g["value_commitments"][0])


# each case: setup(ctx, rnd, owned) -> the call to measure (handles it creates go to `owned`, closed after the test);
# expected per-kernel counts, and the expected Context.launches delta when it differs from their sum (graph path)
def c_msm(ctx, rnd, owned):
    s, p = scalars(rnd, 64), points(ctx, rnd, 64)
    return lambda: ctx.msm(s, p)


def c_msm_batch(ctx, rnd, owned):
    s, p = scalars(rnd, 100), points(ctx, rnd, 100)
    return lambda: ctx.msm_batch(s, p, [0, 5, 5, 40, 100])


def c_points_create(ctx, rnd, owned):
    import bulletproofs_b200 as bp
    p = points(ctx, rnd, 32)
    return lambda: owned.append(bp.PointSet(ctx, p))


def c_points_msm(ctx, rnd, owned):
    import bulletproofs_b200 as bp
    ps = bp.PointSet(ctx, points(ctx, rnd, 32)); owned.append(ps)
    s = scalars(rnd, 60)
    return lambda: ps.msm(s, 3, 20)


def c_points_msm_again(ctx, rnd, owned):      # the term -> point map of the previous call is reused
    call = c_points_msm(ctx, rnd, owned)
    call()
    return call


def c_indexed_msm(ctx, rnd, owned):
    import bulletproofs_b200 as bp
    gens = bp.Gens(ctx, 16, 2); owned.append(gens)
    s, dyn = scalars(rnd, 7), points(ctx, rnd, 3)
    idx = (ctypes.c_uint32 * 7)(1, 0, 2 + 16 + 3, 2 + 2 * 16 + 7, DYN | 0, DYN | 2, 1)
    offs = (ctypes.c_uint64 * 3)(0, 2, 7)
    outs, st = ctypes.create_string_buffer(64), ctypes.create_string_buffer(2)
    return lambda: ctx._check(bp.lib().bp_msm_indexed_batch(ctx._h, gens._h, s, idx, dyn, 3, offs, 2, outs, st))


def c_decompress(ctx, rnd, owned):
    p = points(ctx, rnd, 8)
    return lambda: ctx.decompress(p)


def c_compress(ctx, rnd, owned):
    xyzt = b"".join(ctx.decompress(points(ctx, rnd, 8))[0])
    return lambda: ctx.compress(xyzt)


def c_from_uniform(ctx, rnd, owned):
    u = rnd.randbytes(64 * 8)
    return lambda: ctx.from_uniform_bytes(u)


def c_gens_create(ctx, rnd, owned):
    import bulletproofs_b200 as bp
    return lambda: owned.append(bp.Gens(ctx, 16, 2))


def c_gens_get(ctx, rnd, owned):
    import bulletproofs_b200 as bp
    gens = bp.Gens(ctx, 16, 2); owned.append(gens)
    return lambda: gens.get(1, 1, 3)


class Session:
    """a bp_ipp / bp_ippx handle, ended with the test"""
    def __init__(self, end):
        self.h, self.end = ctypes.c_void_p(), end

    def close(self):
        if self.h:
            self.end(self.h)


def ipp_setup(ctx, rnd, owned, begin):
    import bulletproofs_b200 as bp
    L, N = bp.lib(), 8
    G, H, Q = points(ctx, rnd, N), points(ctx, rnd, N), points(ctx, rnd, 1)
    s = Session(L.bp_ipp_end); owned.append(s)
    call = lambda: ctx._check(L.bp_ipp_begin_points(ctx._h, G, H, N, Q, ctypes.byref(s.h)))
    if begin:
        call()
    return L, s, call


def c_ipp_begin_points(ctx, rnd, owned):
    return ipp_setup(ctx, rnd, owned, False)[2]


def c_ipp_lr(ctx, rnd, owned):
    L, s, _ = ipp_setup(ctx, rnd, owned, True)
    sL, sR, out = scalars(rnd, 9), scalars(rnd, 9), [ctypes.create_string_buffer(32) for _ in range(2)]
    return lambda: ctx._check(L.bp_ipp_lr(s.h, 4, sL, sR, out[0], out[1]))


def c_ipp_fold(ctx, rnd, owned):
    L, s, _ = ipp_setup(ctx, rnd, owned, True)
    f = [scalars(rnd, 4) for _ in range(4)]
    return lambda: ctx._check(L.bp_ipp_fold(s.h, 4, f[0], f[1], f[2], f[3], 1))


def ippx_setup(ctx, rnd, owned, begin, rounds=0):
    import bulletproofs_b200 as bp
    L, N, B = bp.lib(), 2, 2
    G, H, Q = points(ctx, rnd, N), points(ctx, rnd, N), points(ctx, rnd, B)
    Gf, Hf, a, b = (scalars(rnd, B * N) for _ in range(4))
    s = Session(L.bp_ippx_end); owned.append(s)
    call = lambda: ctx._check(L.bp_ippx_begin_points(ctx._h, G, H, N, B, Q, Gf, Hf, a, b, ctypes.byref(s.h)))
    if begin:
        call()
    lr, u, u_inv = ctypes.create_string_buffer(64 * B), scalars(rnd, B), scalars(rnd, B)
    for _ in range(rounds):
        ctx._check(L.bp_ippx_round(s.h, lr)); ctx._check(L.bp_ippx_fold(s.h, u, u_inv))
    return L, s, call, lr, u, u_inv


def c_ippx_begin_points(ctx, rnd, owned):
    return ippx_setup(ctx, rnd, owned, False)[2]


def c_ippx_round(ctx, rnd, owned):
    L, s, _, lr, _, _ = ippx_setup(ctx, rnd, owned, True)
    return lambda: ctx._check(L.bp_ippx_round(s.h, lr))


def c_ippx_fold(ctx, rnd, owned):
    L, s, _, lr, u, u_inv = ippx_setup(ctx, rnd, owned, True)
    ctx._check(L.bp_ippx_round(s.h, lr))
    return lambda: ctx._check(L.bp_ippx_fold(s.h, u, u_inv))


def c_ippx_finish(ctx, rnd, owned):
    L, s, _, _, _, _ = ippx_setup(ctx, rnd, owned, True, rounds=1)
    ab = ctypes.create_string_buffer(128)
    return lambda: ctx._check(L.bp_ippx_finish(s.h, ab))


def c_verify_reject(ctx, rnd, owned):
    """direct path (profiling on): the combined check of the batch fails, so the chunk level and the per-proof level run"""
    import bulletproofs_b200 as bp
    label, proof, V = golden_rangeproof()
    gens = bp.Gens(ctx, 64, 8); owned.append(gens)
    bad = bytearray(proof); bad[140] ^= 1
    proofs = proof + bytes(bad)

    def call():
        assert bp.verify_batch(ctx, gens, bp.Transcript(label), proofs, V * 2, 64, 1, 2) == [0, 1]
    return call


def c_verify_graph(ctx, rnd, owned):
    """reserved geometry: run_device replays the captured graph (profiling off: only the launch total is visible)"""
    import torch
    import bulletproofs_b200 as bp
    label, proof, V = golden_rangeproof()
    gens = bp.Gens(ctx, 64, 8); owned.append(gens)
    ctx.prof_enable(False)
    ver = bp.BatchVerifier(ctx, gens, bp.Transcript(label), 64, 1, 2)
    d_proofs = torch.tensor(list(proof * 2), dtype=torch.uint8, device="cuda")
    d_V = torch.tensor(list(V * 2), dtype=torch.uint8, device="cuda")
    d_verdicts = torch.full((2,), -1, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()

    def call():
        ver.run_device(d_proofs.data_ptr(), d_V.data_ptr(), d_verdicts.data_ptr())
        ctx.synchronize()
        assert d_verdicts.tolist() == [0, 0]
    return call


CHAIN = 5 + 1        # k_rp_decompress, k_rp_transcript, k_rp_head_seq, k_rp_scalars_sum, k_rp_static_sum + k_rp_verdict_batch
CASES = {
    "msm": (c_msm, Counter(k_decompress=1, small_kernels=2, k_compress=1) + PASS),
    "msm_batch_ragged": (c_msm_batch, Counter(k_decompress=1, small_kernels=2, k_compress=1) + PASS),
    "points_create": (c_points_create, Counter(k_decompress=1)),
    "points_msm": (c_points_msm, Counter(small_kernels=3, k_compress=1) + PASS),
    "points_msm_again": (c_points_msm_again, Counter(small_kernels=2, k_compress=1) + PASS),
    "indexed_msm": (c_indexed_msm, Counter(k_decompress=1, small_kernels=1, k_compress=1) + PASS),
    "decompress": (c_decompress, Counter(k_decompress=1)),
    "compress": (c_compress, Counter(k_compress=1)),
    "from_uniform": (c_from_uniform, Counter(k_from_uniform=1)),
    "gens_create": (c_gens_create, Counter(k_from_uniform=1, k_decompress=1)),
    "gens_get": (c_gens_get, Counter(small_kernels=1)),
    "ipp_begin_points": (c_ipp_begin_points, Counter(k_decompress=1)),
    "ipp_lr": (c_ipp_lr, Counter(k_compress=1) + PASS),
    "ipp_fold": (c_ipp_fold, Counter(k_ipp_fold=2)),
    "ippx_begin_points": (c_ippx_begin_points, Counter(k_decompress=2, small_kernels=2)),
    "ippx_round": (c_ippx_round, Counter(small_kernels=2, k_compress=1) + PASS),
    "ippx_fold": (c_ippx_fold, Counter(k_ipp_fold=1)),
    "ippx_finish": (c_ippx_finish, Counter(small_kernels=1)),
    # maps of the new geometry (2) + the chain; fallback level 1: rows, offsets, one pass, chunk verdicts; the per-proof static
    # scalars (k_rp_scalars); level 2: expand, point map, offsets, one pass, proof verdicts
    "verify_reject": (c_verify_reject, Counter(small_kernels=2 + 1 + 3 + 4, k_rp_decompress=1, k_rp_transcript=1, k_rp_head=1, k_rp_scalars=2,
                                               k_rp_static_reduce=1) + PASS + PASS + PASS),
    "verify_graph": (c_verify_graph, Counter(), CHAIN + sum(PASS.values())),
}


@pytest.mark.parametrize("case", list(CASES))
def test_launches_of_one_call(built, case):
    import bulletproofs_b200 as bp
    setup, want, *total = CASES[case]
    ctx = bp.Context(0)                     # fresh: cached geometry (term -> point maps, graphs) must not leak between cases
    owned = []
    try:
        ctx.prof_enable(True)
        call = setup(ctx, random.Random(case), owned)
        ctx.prof_report()                   # drop what the setup launched
        l0 = ctx.launches
        call()
        got = Counter({name: n for name, (_, n) in ctx.prof_report().items()})
        assert got == want
        assert ctx.launches - l0 == (total[0] if total else sum(want.values()))
    finally:
        for h in reversed(owned):
            h.close()
        ctx.close()
