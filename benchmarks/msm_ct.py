"""Constant-time indexed MSM (bp_msm_indexed_batch_ct) against the variable-time bp_msm_indexed_batch, and what routing the provers'
secret commitments through it costs.  Prints the card name and power limit, then one JSON line per measurement.

  python benchmarks/msm_ct.py                  ct vs vartime at the prover's shapes; prove_many (64,1) x 1024 and a 2^16-multiplier R1CS prove
  python benchmarks/msm_ct.py --lib-dir DIR    the prover timings only, with libbpmsm.so / libbulletproofs_host.so from DIR (e.g. a build
                                               of another commit, for a before/after comparison in one session)
  python benchmarks/msm_ct.py --zero-vs-random median per-call time of all-zero against random scalars on both paths (informative only:
                                               a host-clock difference at this resolution is not evidence either way)

Times are host clock around calls that synchronise (H2D, kernels, D2H), median of --reps after --warmup calls."""
import argparse
import json
import os
import random
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bulletproofs_b200 as bp  # noqa: E402
from oracle_binding import L_ORDER as L  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout
        return out.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        return "unknown"


def timed(fn, warmup, reps):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter(); fn(); ts.append(time.perf_counter() - t0)
    return statistics.median(ts)


def shapes(gens):
    """(name, scalars count, point_idx, offsets) at the prover's shapes"""
    rnd = random.Random(1)
    out = [("1024 x 2 (Pedersen commitments)", [1, 0] * 1024, list(range(0, 2049, 2)))]
    row = [0] + [gens.slot_G(0, i) for i in range(64)] + [gens.slot_H(0, i) for i in range(64)]
    out.append(("1024 x 129 (A or S of (64,1) proofs)", row * 1024, list(range(0, 1024 * 129 + 1, 129))))
    s = []
    for j in range(16):
        s += [0] + [gens.slot_G(0, 64 * j + i) for i in range(64)] + [gens.slot_H(0, 64 * j + i) for i in range(64)]
    out.append(("2064 (S of a (64,16) proof)", s, [0, 2064]))
    n = (1 << 17) + 1
    out.append(("2^17 + 1 (R1CS A_I at 2^16 multipliers)", [rnd.randrange(2 + 2 * gens.gens_capacity) for _ in range(n)], [0, n]))
    return out


def msm_compare(ctx, args):
    gens = bp.Gens(ctx, 1 << 16, 1)
    rnd = random.Random(2)
    for name, idx, offs in shapes(gens):
        sc = b"".join(rnd.randrange(L).to_bytes(32, "little") for _ in range(len(idx)))
        st_ct, r_ct = gens.msm_indexed(sc, idx, offs, constant_time=True)
        st_vt, r_vt = gens.msm_indexed(sc, idx, offs)
        assert st_ct == st_vt and r_ct == r_vt, name
        t_ct = timed(lambda: gens.msm_indexed(sc, idx, offs, constant_time=True), args.warmup, args.reps)
        t_vt = timed(lambda: gens.msm_indexed(sc, idx, offs), args.warmup, args.reps)
        print(json.dumps({"shape": name, "terms": len(idx), "n_msm": len(offs) - 1, "ct_ms": round(1e3 * t_ct, 3), "vartime_ms": round(1e3 * t_vt, 3),
                          "ct_over_vartime": round(t_ct / t_vt, 2)}), flush=True)
    gens.close()


def zero_vs_random(ctx, args):
    gens = bp.Gens(ctx, 1 << 16, 1)
    rnd = random.Random(3)
    for name, idx, offs in shapes(gens)[:3]:
        zero = bytes(32 * len(idx))
        rand = b"".join(rnd.randrange(L).to_bytes(32, "little") for _ in range(len(idx)))
        row = {"shape": name}
        for ct in (True, False):
            for label, sc in (("zero", zero), ("random", rand)):
                row[f"{'ct' if ct else 'vartime'}_{label}_ms"] = round(1e3 * timed(lambda: gens.msm_indexed(sc, idx, offs, constant_time=ct), args.warmup, args.reps), 3)
        print(json.dumps(row), flush=True)
    gens.close()


def provers(ctx, args, tag):
    rnd = random.Random(4)
    gens = bp.Gens(ctx, 64, 1)
    B = 1024
    vals = [rnd.randrange(1 << 64) for _ in range(B)]
    bl = b"".join(rnd.randrange(L).to_bytes(32, "little") for _ in range(B))
    seeds = rnd.randbytes(32 * B)
    run = lambda: bp.prove_many(ctx, gens, bp.Transcript(b"msm_ct bench"), vals, bl, 64, 1, seeds)
    st, proofs, _ = run()
    assert all(s == 0 for s in st)
    t = timed(run, 1, args.reps)
    print(json.dumps({"build": tag, "workload": "prove_many (64,1) x 1024", "s": round(t, 4), "proofs_per_s": round(B / t, 1)}), flush=True)
    gens.close()
    k = 32769                                                             # 2 (k - 1) = 2^16 multipliers
    cap = 1 << 16
    gens = bp.Gens(ctx, cap, 1)
    inp = [rnd.randrange(1 << 64) for _ in range(k)]; out = inp[:]; rnd.shuffle(out)
    bl = b"".join(rnd.randrange(L).to_bytes(32, "little") for _ in range(2 * k))

    def tr():
        t = bp.Transcript(b"ShuffleBenchmark"); t.append_message(b"dom-sep", b"ShuffleProof"); t.append_u64(b"k", k); return t
    run = lambda: bp.r1cs_prove(ctx, gens, tr(), bp.GADGET_SHUFFLE, inp + out, bl)
    rc, proof, V = run()
    assert rc == 0 and bp.r1cs_verify(ctx, gens, tr(), bp.GADGET_SHUFFLE, V, proof) == 0
    t = timed(run, 0, max(2, args.reps // 2))
    print(json.dumps({"build": tag, "workload": "R1CS shuffle prove, 2^16 multipliers", "s": round(t, 4)}), flush=True)
    gens.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib-dir", default=None)
    ap.add_argument("--zero-vs-random", action="store_true")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    tag = "this tree"
    if args.lib_dir:
        bp.LIB_PATH = os.path.join(args.lib_dir, "libbpmsm.so")
        bp.HOST_LIB_PATH = os.path.join(args.lib_dir, "libbulletproofs_host.so")
        import ctypes
        have = ctypes.CDLL(bp.LIB_PATH)
        for name in [n for n in bp.SYMBOLS if not hasattr(have, n)]:        # a build that predates an entry point
            del bp.SYMBOLS[name]
        tag = args.lib_dir
    print(json.dumps({"card": card()}), flush=True)
    ctx = bp.Context(0)
    if args.zero_vs_random:
        zero_vs_random(ctx, args)
    else:
        if not args.lib_dir:
            msm_compare(ctx, args)
        provers(ctx, args, tag)
    ctx.close()


if __name__ == "__main__":
    main()
