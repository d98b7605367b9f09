"""bench.py is the driver's entry point: keep it importable and its reference arm runnable without a GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_help_parses():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    for flag in ("--gpus", "--steps", "--warmup", "--impl", "--dump-outputs"):
        assert flag in r.stdout


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "proofs/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["e2e"]["h2d_bytes_per_step"] == 0


def test_msm_workload_reference_arm():
    """BASELINE config 4's CPU arm (`--workload msm --impl reference`) runs without a GPU and prints one JSON line in terms/s."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "msm", "--lg", "10", "--msms", "2", "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "terms/s" and d["value"] > 0 and d["config"]["lg_n"] == 10


def test_dump_outputs_only_on_the_gpu_rangeproof_path(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path / "out")],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and not (tmp_path / "out").exists()


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_timed_step(tmp_path):
    out = tmp_path / "out"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1", "--streams", "2", "--group", "2",
                        "--batch", "64", "--no-cpu-baseline", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.strip()][-1])
    assert d["steps"] == 3 and d["config"]["proofs_per_step"] == 2 * 2 * 64
    verdicts, batch_ok = np.load(out / "verdicts.npy"), np.load(out / "batch_ok.npy")
    assert sorted(p.name for p in out.iterdir()) == ["batch_ok.npy", "verdicts.npy"]
    assert verdicts.dtype == np.float32 and verdicts.shape == (2, 2 * 64) and not verdicts.any()
    assert batch_ok.dtype == np.float32 and batch_ok.shape == (2, 2) and (batch_ok == 1).all()


def test_both_arms_emit_the_same_config():
    """the driver compares the two arms' `config` objects: same keys, same values"""
    sys.path.insert(0, ROOT)
    import argparse
    import bench
    args = argparse.Namespace(batch=1024, m=1, group=8, streams=8)
    a, b = bench.make_config(args, 1), bench.make_config(args, 1)
    assert a == b and set(a) >= {"workload", "n", "m", "batch", "batches_per_group", "groups_in_flight", "proofs_per_step", "l2", "parallelism"}
