#!/usr/bin/env python
"""bench.py — batched 64-bit range-proof verifications/sec (BASELINE.json metric) on N B200s.

Workload (config.workload): BASELINE config 2, batches of 1024 independent 64-bit RangeProofs (m = 1, 672 B proof + 32 B
commitment each).  Every batch is verified on its own: transcript replay + verification scalars + 17 408 Ristretto
decompressions + one 17 538-term random-linear-combination MSM + identity check -> 1024 verdicts and one accept flag.
The engine launches batches in *groups* (`--group` batches share one launch sequence so that the grids fill the 148 SMs)
and keeps `--streams` groups in flight.

One *step* = one sweep over all in-flight groups = streams x group batches (config.proofs_per_step); the timed region is
exactly `--steps` such sweeps after `--warmup` untimed ones.  Every arena is reserved and every launch graph captured and
run once in the verifier constructors, before any timed region, whatever --warmup is.

  value  : whole-job proofs/s with the input batches already resident in HBM (device-pointer entry point), CUDA events,
           max over ranks
  e2e    : the same metric through the host-buffer C-ABI call (pinned host buffers; the H2D copy of the proofs and the
           D2H copy of the verdicts are inside the timed region)
  --impl reference : the reference's CPU path (the oracle restatement, fastest vector backend the host has; the Rust
           crate cannot be built in this image) on all host cores, same metric and config.
  --workload msm --lg K : BASELINE config 4, batched Ristretto MSMs of 2^K terms (whole MSMs per rank).
  --dump-outputs DIR : after the timed steps, rank 0 writes what the device-resident path returned in its last timed step
           (per-proof verdict codes, per-batch accept flags) as DIR/<name>.npy in float32.  The inputs depend only on the
           arguments, so two builds can be compared output for output.

Inputs rotate through a pool of distinct groups larger than L2 (config.l2 says so).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

# one hardware work queue per stream (the default of 8 makes >8 streams share queues and serialise)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
# the benchmark may run from a read-only tree and writes nothing into it
sys.dont_write_bytecode = True

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

N_BITS = 64
LABEL = b"AggregateRangeProofBenchmark"            # benches/range_proof.rs:34
L2_BYTES = 126 * 1024 * 1024
METRIC = "64-bit rangeproof verifications/sec (batched)"
INT_PEAK = 9.25e12                                 # IMAD.WIDE.U32 thread-level multiply-adds/s, measured (profiles/r1_imad_peak.md)


def effective_cores():
    """host cores this process may actually use: min(affinity, cgroup cpu.max quota)"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


def parse_cpulist(text):
    out = set()
    for part in text.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        out.update(range(int(a), int(b or a) + 1))
    return out


def pin_to_gpu_numa_node(local, world_local):
    """Bind this rank's threads to the CPUs of its GPU's NUMA node (and to this rank's slice of them when several local ranks
    share a node).  Returns a short description for the JSON line; never fails the run."""
    try:
        import torch
        prop = torch.cuda.get_device_properties(local)
        bus = f"{prop.pci_domain_id:04x}:{prop.pci_bus_id:02x}:{prop.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return {"numa_node": None}
        cpus = sorted(parse_cpulist(open(f"/sys/devices/system/node/node{node}/cpulist").read()) & os.sched_getaffinity(0))
        if not cpus:
            return {"numa_node": node, "pinned": 0}
        # local ranks on the same node split its CPUs
        peers = []
        for r in range(world_local):
            p = torch.cuda.get_device_properties(r)
            b = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
            try:
                if int(open(f"/sys/bus/pci/devices/{b}/numa_node").read()) == node:
                    peers.append(r)
            except Exception:
                pass
        if local in peers and len(peers) > 1 and len(cpus) >= 2 * len(peers):
            per = len(cpus) // len(peers); i = peers.index(local)
            cpus = cpus[i * per:(i + 1) * per]
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "pinned": len(cpus)}
    except Exception as e:                                     # pragma: no cover - best effort
        return {"numa_node": None, "error": str(e)[:80]}


def make_workload(count, rank, m_parties):
    """Synthetic input: `count` valid (64,m) proofs over uniform 64-bit values and uniform blindings.
    The proofs are produced by the CPU oracle's prover (test infrastructure used as a data generator only;
    nothing on the measured path touches it)."""
    import random
    from oracle_binding import Oracle, L_ORDER
    orc = Oracle()
    og = orc.gens(N_BITS, m_parties)
    rnd = random.Random(1000 + rank)
    values = [rnd.randrange(1 << N_BITS) for _ in range(count * m_parties)]
    blind = b"".join(rnd.randrange(L_ORDER).to_bytes(32, "little") for _ in range(count * m_parties))
    seeds = b"".join((rank * count + i).to_bytes(8, "little") + bytes(24) for i in range(count))
    proofs, Vs = orc.prove_many(og, orc.transcript(LABEL), values, blind, N_BITS, m_parties, seeds, nthreads=effective_cores())
    return orc, og, proofs, Vs


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed regions (B200_PROFILING.md recipe): ONE `nvidia-smi -lms 50`
    process for all GPUs of the job (rank 0 owns it), every line stamped on arrival; stop() summarises the samples that fell
    inside mark_begin()..mark_end() windows."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, indices):
        super().__init__(daemon=True)
        self.indices, self.samples, self.windows, self.proc = list(indices), [], [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", ",".join(map(str, self.indices)), "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                f = [x.strip() for x in line.split(",")]
                if len(f) >= 8:
                    self.samples.append((time.perf_counter(), f))
        except Exception:
            pass

    def mark_begin(self):
        self.windows.append([time.perf_counter(), None])

    def mark_end(self):
        self.windows[-1][1] = time.perf_counter()

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=3)
        inside = [f for t, f in self.samples if any(a <= t <= (b or 1e30) for a, b in self.windows)] or [f for _, f in self.samples]
        sm = sorted(int(float(f[1])) for f in inside)
        reasons = set()
        for f in inside:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(float(inside[0][2])) if inside else None,
                "reasons": sorted(reasons), "samples": len(sm), "gpus_sampled": len(self.indices), "power_w_max": max((float(f[3]) for f in inside), default=None)}


def make_config(args, world):
    """identical keys and values in both arms (the driver compares them)"""
    per_step = args.streams * args.group * args.batch
    return {"workload": f"batched verify of {args.batch}x 64-bit RangeProofs (m={args.m}) per batch; {args.group} batches per launch group, {args.streams} groups in flight per GPU",
            "n": N_BITS, "m": args.m, "batch": args.batch, "batches_per_group": args.group, "groups_in_flight": args.streams,
            "step": f"one sweep over the in-flight groups = {args.streams * args.group} batches = {per_step} proofs per GPU",
            "proofs_per_step": per_step * world,
            "l2": "inputs larger than L2: a pool of distinct input groups (> 126 MiB) is cycled",
            "parallelism": f"independent batches per GPU x{world}; one NCCL broadcast of the generator table, no data-path collective"}


def cpu_backend_survey(orc, og, t, proofs, plen, Vs, m):
    """single-thread us per (64,m) verification on every MSM field backend of the oracle this CPU supports (u64 serial, the
    reference's default 4-way avx2 backend, 4-way avx512ifma); selects the fastest and returns {backend: us}."""
    out = {}
    for name in ("u64", "avx2", "ifma"):
        if orc.set_backend(name) != 0:
            continue
        orc.verify_many(og, t, proofs[:4 * plen], plen, Vs[:4 * 32 * m], N_BITS, m, 4, nthreads=1)
        t0 = time.perf_counter(); n1 = 0
        while time.perf_counter() - t0 < 0.8:
            st = orc.verify_many(og, t, proofs[:8 * plen], plen, Vs[:8 * 32 * m], N_BITS, m, 8, nthreads=1); n1 += 8
            assert not any(st)
        out[name] = round(1e6 * (time.perf_counter() - t0) / n1, 1)
    best = min(out, key=out.get)
    orc.set_backend(best)
    return out


def cpu_rlc_line(orc, og, t, proofs, plen, Vs, m, batch, cores):
    """The apples-to-apples CPU line: the same random-linear-combination batch the GPU engine runs (the reference has no batch
    verifier), one combined Pippenger MSM per thread's chunk of the batch, on all host cores."""
    st = orc.verify_rlc(og, t, proofs, plen, Vs, N_BITS, m, batch, nthreads=cores)
    assert not any(st)
    done, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < 4.0:
        orc.verify_rlc(og, t, proofs, plen, Vs, N_BITS, m, batch, nthreads=cores); done += batch
    dt = time.perf_counter() - t0
    return {"value": done / dt, "unit": "proofs/s", "cores": cores, "note": f"{batch}-proof batch split in {cores} chunks, one combined MSM per chunk; not part of the reference (SURVEY.md 8a row A6)"}


def run_reference(args, rank, world):
    """The reference's own CPU path for the metric: per-proof RangeProof::verify_multiple on every host core (oracle
    restatement with the fastest field backend the host supports, kind "port").  Rank 0 only; a bounded sample of the step."""
    if rank != 0:
        return
    cores = effective_cores()
    batch, m = args.batch, args.m
    orc, og, proofs, Vs = make_workload(batch, 0, m)
    plen = len(proofs) // batch
    t = orc.transcript(LABEL)
    backends = cpu_backend_survey(orc, og, t, proofs, plen, Vs, m)        # leaves the fastest backend selected
    backend = orc.backend_name()
    probe = min(batch, 8 * cores)
    t0 = time.perf_counter(); st = orc.verify_many(og, t, proofs[:probe * plen], plen, Vs[:probe * 32 * m], N_BITS, m, probe, nthreads=cores); dt = time.perf_counter() - t0
    assert not any(st)
    rate = probe / dt
    budget_s = 90.0
    sample = int(max(cores, min(batch, rate * budget_s / max(1, args.steps + args.warmup))))
    for _ in range(args.warmup):
        orc.verify_many(og, t, proofs[:sample * plen], plen, Vs[:sample * 32 * m], N_BITS, m, sample, nthreads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        st = orc.verify_many(og, t, proofs[:sample * plen], plen, Vs[:sample * 32 * m], N_BITS, m, sample, nthreads=cores)
    dt = time.perf_counter() - t0
    assert not any(st)
    value = sample * args.steps / dt
    terms = 2 * N_BITS * m + 2 * ((N_BITS * m).bit_length() - 1) + m + 6
    cpu = {"value": value, "unit": "proofs/s", "cores": cores, "kind": "port", "backend": backend,
           "single_thread_us_per_verify": backends,      # every field backend this host supports, same proofs (the arm runs the fastest)
           "published_reference_us_per_verify": {"avx2_i7_7800X_3.5GHz": 1040, "u64": 1490, "ifma": "about 1.5x faster than avx2", "source": "README.md:76-84"},
           "rlc_batch": cpu_rlc_line(orc, og, t, proofs, plen, Vs, m, batch, cores),
           "sample": f"{sample} of the step's (64,{m}) proofs per step, per-proof verify_multiple ({terms} terms), one proof per task on {cores} threads"}
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": value, "unit": "proofs/s", "n_gpus": 0,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
                      "vs_baseline": None, "dtype": f"{backend} (CPU)", "data": "synthetic (oracle-proved valid proofs over uniform 64-bit values)",
                      "config": make_config(args, max(1, args.gpus)),
                      "cpu_baseline": cpu, "e2e": {"value": value, "unit": "proofs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--streams", type=int, default=8, help="launch groups in flight (one context + stream each)")
    ap.add_argument("--group", type=int, default=8, help="batches per launch group")
    ap.add_argument("--threads", type=int, default=0, help="host threads issuing groups; 0 = min(2, host cores per rank)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--m", type=int, default=1, help="parties per proof (BASELINE config 3: --m 16 --batch 256); the bench line is the default")
    ap.add_argument("--batch", type=int, default=1024, help="proofs per verified batch")
    ap.add_argument("--workload", default="rangeproof", choices=["rangeproof", "msm"])
    ap.add_argument("--lg", type=int, default=16, help="--workload msm: terms per MSM = 2^lg")
    ap.add_argument("--msms", type=int, default=8, help="--workload msm: MSMs per call")
    ap.add_argument("--window", type=int, default=0, help="--workload msm: fix the Pippenger window (bits); 0 = by size")
    ap.add_argument("--check-lg", type=int, default=16, help="--workload msm: compare the first MSM with the CPU oracle up to this size")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's verdicts and batch accept flags as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.dump_outputs and (args.workload != "rangeproof" or args.impl != "ours"):
        ap.error("--dump-outputs applies to the GPU range-proof workload")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    if args.workload == "msm":
        import bench_msm
        return bench_msm.main(args, rank, world, local, local_world)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import bulletproofs_b200 as bp

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback on the MSM path")
    torch.cuda.set_device(local)
    pin = pin_to_gpu_numa_node(local, local_world)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    M, BATCH, G, S = args.m, args.batch, max(1, args.group), max(1, args.streams)
    orc, og, proofs, Vs = make_workload(BATCH, rank, M)
    plen = len(proofs) // BATCH
    streams = [torch.cuda.Stream(device=local) for _ in range(S)]
    ctxs = [bp.Context(local, stream=s.cuda_stream) for s in streams]

    # generator table: derived once on rank 0, one NCCL broadcast over NVLink, imported by every context's table
    gens0 = bp.Gens(ctxs[0], N_BITS, M, empty=(rank != 0))
    _, table_bytes = gens0.device_table()
    table = torch.empty(table_bytes, dtype=torch.uint8, device="cuda")
    if rank == 0:
        gens0.table_export(table.data_ptr())
    from bulletproofs_b200.dist import broadcast_table
    broadcast_table(table, src=0)                  # the path's only collective: one NCCL broadcast over NVLink
    torch.cuda.synchronize()
    gens = [gens0]
    if rank != 0:
        gens0.table_import(table.data_ptr())
    for c in ctxs[1:]:
        g = bp.Gens(c, N_BITS, M, empty=True); g.table_import(table.data_ptr()); gens.append(g)
    assert gens[-1].G(0, 5) == orc.gens_get(og, 0, 0, 5)

    transcript = bp.Transcript(LABEL)
    # the constructor reserves the geometry: arenas, maps, the captured launch graph and one warm pass -- nothing allocates later
    ver = [bp.BatchVerifier(ctxs[i], gens[i], transcript, N_BITS, M, BATCH, G) for i in range(S)]

    # input pool larger than L2: rotations of the proof order (distinct memory, same proofs); one pool entry = one group of G batches
    group_bytes = G * BATCH * (plen + 32 * M)
    P = L2_BYTES // group_bytes + 2
    pr = np.frombuffer(proofs, dtype=np.uint8).reshape(BATCH, plen); vs = np.frombuffer(Vs, dtype=np.uint8).reshape(BATCH, 32 * M)
    h_proofs = torch.empty((P, G, BATCH, plen), dtype=torch.uint8).pin_memory(); h_vs = torch.empty((P, G, BATCH, 32 * M), dtype=torch.uint8).pin_memory()
    for i in range(P):
        for j in range(G):
            sh = (i * G + j) * 5
            h_proofs[i, j] = torch.from_numpy(np.roll(pr, sh, axis=0).copy()); h_vs[i, j] = torch.from_numpy(np.roll(vs, sh, axis=0).copy())
    d_proofs = h_proofs.cuda(); d_vs = h_vs.cuda()
    d_verdicts = torch.zeros((S, G * BATCH), dtype=torch.int32, device="cuda")
    h_ok = torch.zeros((S, G), dtype=torch.int32).pin_memory()
    torch.cuda.synchronize()

    # correctness gate before timing: GPU verdicts == expected on a group with one damaged proof in one batch
    gp = bytearray(h_proofs[1].numpy().tobytes()); bad_at = (G - 1) * BATCH + 7; gp[bad_at * plen + 300] ^= 1
    got, ok = bp.verify_group(ctxs[0], gens[0], transcript, bytes(gp), h_vs[1].numpy().tobytes(), N_BITS, M, BATCH, G)
    assert [i for i, v in enumerate(got) if v] == [bad_at] and ok == [1] * (G - 1) + [0], "GPU verdicts differ from the expected ones"

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    from concurrent.futures import ThreadPoolExecutor
    NT = args.threads if args.threads > 0 else min(2, max(1, effective_cores() // max(1, local_world)))
    NT = max(1, min(NT, S))
    pool = ThreadPoolExecutor(NT) if NT > 1 else None

    def run_sweeps(group_fn, first, n):
        """sweeps first..first+n-1; in every sweep each context k launches one group; thread t drives the contexts with k % NT == t"""
        def worker(t):
            for i in range(first, first + n):
                for k in range(t, S, NT):
                    group_fn(i, k)
        if pool is None:
            worker(0)
        else:
            list(pool.map(worker, range(NT)))

    def timed(group_fn, drain_fn, steps, warmup):
        run_sweeps(group_fn, 0, warmup)
        drain_fn()
        barrier()                                      # outside the measured window
        l0 = sum(c.launches for c in ctxs)
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ends = [torch.cuda.Event() for _ in range(S)]
        t0 = time.perf_counter()
        start.record(streams[0])
        for s in streams[1:]:
            s.wait_event(start)
        run_sweeps(group_fn, warmup, steps)
        host_issue = time.perf_counter() - t0
        drain_fn()
        for s, e in zip(streams, ends):
            e.record(s); streams[0].wait_event(e)
        end.record(streams[0])
        end.synchronize()
        wall = time.perf_counter() - t0                # this rank's own window: no barrier, no collective inside
        ms = start.elapsed_time(end)
        launches = sum(c.launches for c in ctxs) - l0
        times = torch.tensor([ms * 1e-3, wall, host_issue], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(times, op=dist.ReduceOp.MAX)
        ms_max, wall_max, issue_max = (float(x) for x in times.tolist())
        return ms_max * 1e3, wall_max, launches, issue_max

    proofs_per_step = S * G * BATCH

    # ---- value: inputs resident in HBM
    # at most two groups queued per stream (the host-buffer path below has one): a deeper queue only adds driver back-pressure on the issuing threads
    dev_ev = [[torch.cuda.Event(), torch.cuda.Event()] for _ in range(S)]
    dev_cnt = [0] * S

    def group_dev(i, k):
        j = (i * S + k) % P
        e = dev_ev[k][dev_cnt[k] & 1]
        if dev_cnt[k] >= 2:
            e.synchronize()
        ver[k].run_device(d_proofs[j].data_ptr(), d_vs[j].data_ptr(), d_verdicts[k].data_ptr(), h_ok[k].data_ptr())
        e.record(streams[k]); dev_cnt[k] += 1

    clk = None
    if rank == 0:
        clk = ClockSampler(range(local_world)); clk.start()
        time.sleep(0.3)                               # let the sampler come up before the first timed region
        clk.mark_begin()
    ms_dev, _, launches, host_issue_dev = timed(group_dev, lambda: None, args.steps, args.warmup)
    if clk:
        clk.mark_end()
    assert int(h_ok.min()) == 1 and int(d_verdicts.abs().max()) == 0, "a timed batch did not verify"
    if args.dump_outputs and rank == 0:
        # every context's last group is the last timed sweep: verdicts[k] and batch_ok[k] are what context k returned for it
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in (("verdicts", d_verdicts), ("batch_ok", h_ok)):
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), t.cpu().numpy().astype(np.float32))
    value = world * proofs_per_step * args.steps / (ms_dev * 1e-3)

    # ---- e2e: host buffers through the public C-ABI call (H2D + kernels + D2H per group)
    def group_e2e(i, k):
        j = (i * S + k) % P
        if ver[k].busy:
            assert not any(ver[k].finish())
        ver[k].begin(h_proofs[j].data_ptr(), h_vs[j].data_ptr())

    def drain_e2e():
        for v in ver:
            if v.busy:
                assert not any(v.finish())

    if clk:
        clk.mark_begin()
    ms_e2e, wall_e2e, _, host_issue_e2e = timed(group_e2e, drain_e2e, args.steps, args.warmup)
    clocks = None
    if clk:
        clk.mark_end()
        clocks = clk.stop()
    e2e_s = max(ms_e2e * 1e-3, wall_e2e)
    e2e_value = world * proofs_per_step * args.steps / e2e_s
    h2d = S * (G * BATCH * (plen + 32 * M) + 512)
    d2h = S * (4 * G * BATCH + 8 * G)

    # ---- per-kernel durations (CUDA events around every launch of one group, direct launches on a single stream) -> roofline block
    ctxs[0].prof_enable(True)
    psteps = 5
    for i in range(psteps):
        ver[0].run_device(d_proofs[i % P].data_ptr(), d_vs[i % P].data_ptr(), d_verdicts[0].data_ptr(), None)
    prof = ctxs[0].prof_report(); ctxs[0].prof_enable(False)
    total_ms = sum(v[0] for v in prof.values())
    # dominant kernel = the Pippenger bucket accumulation (the MSM kernel north_star names; with the per-proof decompressions the
    # largest consumer of the integer-multiply pipe).  The transcript / window-combination kernels have longer solo durations but
    # are latency chains of a few warps that overlap with the other groups in flight.
    dom = "k_msm_accumulate" if "k_msm_accumulate" in prof else max(prof, key=lambda k: prof[k][0])
    dom_ms = prof[dom][0] / prof[dom][1]
    k_lg = (N_BITS * M).bit_length() - 1
    T_terms = 2 + 2 * N_BITS * M + BATCH * (4 + 2 * k_lg + M)
    alg_bytes_batch = BATCH * (32 * (9 + 2 * k_lg) + 32 * M + 1) + 32 * (2 * N_BITS * M + 2)     # SURVEY.md §8(d), per verified batch
    alg_bytes = G * (64 * T_terms + 32) if dom.startswith("k_msm") else G * alg_bytes_batch       # SURVEY.md §8(d): G MSMs of T terms per launch
    W_win = (255 + 10) // 11; pts = BATCH * (4 + 2 * k_lg + M); Nv = N_BITS * M
    wide = (pts * (257 * 44 + 29 * 72)                      # decompress: one 2^252-3 exponentiation + decode + Niels form per point
            + T_terms * W_win * 7 * 72                       # bucket accumulation: one mixed addition per term and window
            + W_win * (59 * 64 + 1) * 9 * 72                 # bucket reduction: 59 additions per thread, 64 threads per window
            + BATCH * (Nv * 3 + (4 + 2 * k_lg + M) * 3 + 170) * 192)   # scalar assembly (3 products per generator index) + per-proof head
    batches_per_s = value / world / BATCH
    int_pipe = {"unit": "wide multiply-adds/s (IMAD.WIDE.U32, thread level)", "per_batch": wide, "achieved": wide * batches_per_s, "peak": INT_PEAK,
                "frac": wide * batches_per_s / INT_PEAK, "peak_source": "measured, benchmarks/imad_microbench.cu (profiles/r1_imad_peak.md)"}
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("hbm_gbs", 6650.0)
    achieved = alg_bytes / (dom_ms * 1e-3) / 1e9
    ncu = {}
    try:
        ncu = json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")))
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": ncu.get("dram_bytes_per_launch", {}).get(dom),
                "peak_source": "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)",
                "algorithmic_bytes_per_launch": alg_bytes, "units_per_launch": f"{G} MSMs x ({T_terms} terms x 64 B + 32 B)" if dom.startswith("k_msm") else f"{G * BATCH} proofs",
                "kernel_ms": dom_ms, "kernel_share_of_step": prof[dom][0] / total_ms,
                "whole_step": {"algorithmic_bytes_per_batch": alg_bytes_batch, "achieved_GBps_at_value": alg_bytes_batch * batches_per_s / 1e9},
                "int_pipe": int_pipe,
                "note": "integer-pipe bound path (IMAD.WIDE field multiplies): the HBM fraction is reported as BASELINE.json asks; issue-slot / FMA-pipe utilisation per kernel is in profiles/",
                "per_kernel_ms_per_group": {k: round(v[0] / psteps, 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}}
    if ncu.get("fmaheavy_busy_cycles_per_sm_per_group") and clocks and clocks.get("sm_mhz"):
        cyc_per_group = ms_dev / (args.steps * S) * 1e-3 * clocks["sm_mhz"] * 1e6
        int_pipe["ncu_fmaheavy"] = {"busy_cycles_per_sm_per_group": ncu["fmaheavy_busy_cycles_per_sm_per_group"], "frac": ncu["fmaheavy_busy_cycles_per_sm_per_group"] * (G / ncu.get("group", G)) / cyc_per_group,
                                    "source": ncu.get("source")}

    out = {"metric": METRIC, "value": value, "unit": "proofs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32x8 (mod 2^255-19) / u32x8 (mod l)",
           "data": "synthetic (oracle-proved valid proofs over uniform 64-bit values)",
           "config": make_config(args, world),
           "e2e": {"value": e2e_value, "unit": "proofs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": 1e3 * e2e_s / args.steps},
           "gpu_launches": launches, "clocks": clocks, "roofline": roofline,
           "diag": {"host_threads": NT, "host_issue_ms_per_step": round(1e3 * host_issue_dev / args.steps, 4), "host_issue_ms_per_step_e2e": round(1e3 * host_issue_e2e / args.steps, 4),
                    "numa": pin, "input_pool_groups": P, "input_pool_MiB": P * group_bytes >> 20}}

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = effective_cores()
        t = orc.transcript(LABEL)
        backends = cpu_backend_survey(orc, og, t, proofs, plen, Vs, M)
        done, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < 12.0:
            st = orc.verify_many(og, t, proofs, plen, Vs, N_BITS, M, BATCH, nthreads=cores); done += BATCH
            assert not any(st)
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": done / dt, "unit": "proofs/s", "cores": cores, "kind": "port", "backend": orc.backend_name(), "single_thread_us_per_verify": backends,
                               "rlc_batch": cpu_rlc_line(orc, og, t, proofs, plen, Vs, M, BATCH, cores),
                               "sample": f"{done} per-proof verify_multiple calls (the {BATCH}-proof batch x{done // BATCH}) on {cores} threads, {dt:.1f} s"}
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
