"""CPU tier of the constant-time indexed MSM (bulletproofs_b200/csrc/msm_ct.cuh, bp_msm_indexed_batch_ct).

- The recoding, table, lookup and chunked Straus loop, compiled for the host from tests/host_emul/emul_ct.cpp, against the oracle.
- A compile-time audit: the secret-dependent templates instantiated on a word type that cannot be branched on or used as an index,
  plus negative controls that must fail to compile.
- A SASS guard on libbpmsm.so.
- The host mirror's routing, through a call log on the mock engine: the prover's commitments to secrets reach only the ct entry
  point, with point indices and offsets that do not depend on the secrets.
- The symbols of include/bpmsm_ct.h are exported and bound.
"""
import ctypes
import os
import random
import re
import shutil
import subprocess

import pytest

from oracle_binding import L_ORDER as l

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EDGE = [0, 1, 8, 15, 16, l - 1, 2**252, int("08" * 31 + "88", 16), int("0" + "7" * 62 + "8", 16), int("8" * 63, 16) % l, 2**128 - 1, l - 2**200]


def le(x):
    return x.to_bytes(32, "little")


def _gxx():
    return shutil.which("g++")


@pytest.fixture(scope="module")
def E(built, tmp_path_factory):
    """tests/host_emul/emul_ct.cpp built for the host (g++) into a temporary directory"""
    if not _gxx():
        pytest.skip("g++ not available")
    so = str(tmp_path_factory.mktemp("emul_ct") / "libemul_ct.so")
    subprocess.run([_gxx(), "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, os.path.join(ROOT, "tests", "host_emul", "emul_ct.cpp")], check=True)
    lib = ctypes.CDLL(so)
    lib.emul_msm_ct.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.POINTER(ctypes.c_uint64), ctypes.c_uint32, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_char_p]
    return lib


def emul_ct(E, scalars, points, offsets, ch):
    n = len(offsets) - 1
    outs, st = ctypes.create_string_buffer(32 * n), ctypes.create_string_buffer(n)
    assert E.emul_msm_ct(scalars, points, (ctypes.c_uint64 * (n + 1))(*offsets), n, ch, outs, st) == 0
    return list(st.raw), [outs.raw[32 * i:32 * i + 32] for i in range(n)]


def oracle_msms(orc, scalars, points, offsets):
    res = []
    for j in range(len(offsets) - 1):
        a, b = offsets[j], offsets[j + 1]
        if a == b:
            res.append(bytes(32)); continue
        rc, o = orc.msm(scalars[32 * a:32 * b], points[32 * a:32 * b])
        assert rc == 0
        res.append(o)
    return res


def test_recoding_digits(E):
    rnd = random.Random(21)
    for s in EDGE + [rnd.randrange(l) for _ in range(300)]:
        d = (ctypes.c_int8 * 64)()
        E.emul_ct_recode(le(s), d)
        assert all(-8 <= x <= 8 for x in d), s
        assert sum(x * 16**i for i, x in enumerate(d)) == s, s
    d = (ctypes.c_int8 * 64)(); E.emul_ct_recode(le(int("0" + "7" * 62 + "8", 16)), d)
    assert list(d[:63]) == [-8] * 63                     # every digit at the table's edge


def test_canonicality_mask(E):
    rnd = random.Random(22)
    for s, want in [(0, 0), (l - 1, 0), (l, 1), (l + 1, 1), (2**256 - 1, 1), (2**255, 1), (2**252, 0)] + [(rnd.randrange(l), 0) for _ in range(50)] + [(rnd.randrange(l, 2**256), 1) for _ in range(50)]:
        assert E.emul_ct_geq_l(le(s)) == want, hex(s)


@pytest.mark.parametrize("ch", [1, 2, 3, 4, 16])
def test_emulated_ct_msm_matches_oracle(E, orc, ch):
    """random and edge scalars; ragged offsets with empty MSMs, so that chunk boundaries fall inside and across MSMs"""
    rnd = random.Random(23 + ch)
    pool = [orc.from_uniform(rnd.randbytes(64)) for _ in range(12)]
    lens = [1, 2, 3, 0, 5, 17, 4, 0, 33, len(EDGE), 9]
    offsets = [0]
    for n in lens:
        offsets.append(offsets[-1] + n)
    T = offsets[-1]
    sc = [rnd.randrange(l) for _ in range(T)]
    e0 = offsets[lens.index(len(EDGE))]
    sc[e0:e0 + len(EDGE)] = EDGE
    pts = [rnd.choice(pool) for _ in range(T)]
    pts[0:3] = [pool[0]] * 3                           # repeated slots in one MSM
    sc_b, pt_b = b"".join(le(x) for x in sc), b"".join(pts)
    st, got = emul_ct(E, sc_b, pt_b, offsets, ch)
    assert st == [0] * len(lens)
    assert got == oracle_msms(orc, sc_b, pt_b, offsets)


def test_emulated_ct_msm_zero_and_noncanonical(E, orc):
    rnd = random.Random(24)
    pts = b"".join(orc.from_uniform(rnd.randbytes(64)) for _ in range(6))
    st, got = emul_ct(E, bytes(32 * 6), pts, [0, 6], 4)
    assert st == [0] and got == [bytes(32)]              # all-zero scalars: the identity
    sc = [rnd.randrange(l) for _ in range(6)]
    sc_bad = sc[:3] + [l] + sc[4:]
    st, got = emul_ct(E, b"".join(le(x) for x in sc_bad), pts, [0, 3, 6], 2)
    assert st == [0, 3]                                 # only the MSM holding the scalar >= l is flagged
    assert got[0] == orc.msm(b"".join(le(x) for x in sc[:3]), pts[:96])[1]


def test_secret_type_audit_compiles_and_has_teeth(tmp_path):
    """msm_ct.cuh's recoding and selection instantiated on a word type without bool/integer conversion or comparisons compile;
    a branch, an index and a comparison on that type each fail to compile (negative controls)."""
    if not _gxx():
        pytest.skip("g++ not available")
    src = os.path.join(ROOT, "tests", "host_emul", "ct_audit.cpp")
    r = subprocess.run([_gxx(), "-std=c++17", "-fsyntax-only", src], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    for n in (1, 2, 3):
        r = subprocess.run([_gxx(), "-std=c++17", "-fsyntax-only", f"-DCT_AUDIT_NEGATIVE_CONTROL={n}", src], capture_output=True, text=True)
        assert r.returncode != 0, f"negative control {n} compiled: the audit type lets a secret steer control flow or addressing"
        assert "negative_control" in r.stderr or "ct_audit.cpp" in r.stderr


def test_ct_kernels_sass_has_no_local_memory_or_indirect_branch(built):
    """Guard, not a proof: in the SASS of the k_msm_ct_* kernels there is no local-memory access (LDL/STL: a compiler-demoted
    array, the usual way a secret index reaches the address bus) and no indirect branch (BRX/JMX).  Control-flow equivalence and
    the absence of secret-dependent addresses are argued in msm_ct.cuh and checked by the type audit above."""
    cuobjdump = shutil.which("cuobjdump") or ("/usr/local/cuda/bin/cuobjdump" if os.path.exists("/usr/local/cuda/bin/cuobjdump") else None)
    if not cuobjdump:
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([cuobjdump, "-sass", os.path.join(ROOT, "bulletproofs_b200", "libbpmsm.so")], capture_output=True, text=True, check=True).stdout
    funcs = re.split(r"\n\s*Function : ", sass)
    ct = [f for f in funcs if re.match(r"_Z\d+k_msm_ct_", f)]
    assert sorted(re.match(r"_Z\d+(k_msm_ct_\w+?)P", f).group(1) for f in ct) == ["k_msm_ct_recode", "k_msm_ct_reduce", "k_msm_ct_straus", "k_msm_ct_table"]
    for f in ct:
        name = f.split("\n", 1)[0]
        for op in ("LDL", "STL", "BRX", "JMX"):
            assert not re.search(rf"\b{op}\b", f), (name, op)


def test_ct_header_symbols_are_exported_and_bound(built):
    """include/bpmsm_ct.h: every declared entry point is exported by libbpmsm.so and bound in CT_SYMBOLS (apart from SYMBOLS, which
    holds exactly the declarations of bpmsm.h)"""
    import bulletproofs_b200 as bp
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "bpmsm_ct.h")).read(), flags=re.S)
    declared = sorted(set(re.findall(r"\b(bp_[a-z0-9_]+)\s*\(", text)))
    assert declared == sorted(bp.CT_SYMBOLS) == ["bp_msm_indexed_batch_ct"]
    assert not set(bp.CT_SYMBOLS) & set(bp.SYMBOLS)
    L = bp.ct_lib()
    for name in declared:
        assert hasattr(L, name)


# ---------------------------------------------------------------- routing of the host mirror, through a call log
# The C++ mirror, built as the library build builds it (-DBP_HOST_REQUIRE_CT), linked with the mock engine (the oracle's arithmetic
# behind the C ABI) and tests/mock_engine/mock_ct_log.c, which adds the ct entry point and logs every MSM call (the variable-time
# entry points through -Wl,--wrap).  One library, built in a temporary directory.
CT, VT = "bp_msm_indexed_batch_ct", "bp_msm_indexed_batch"


def build_routing_lib(tmp):
    if not (_gxx() and shutil.which("gcc")):
        pytest.skip("gcc / g++ not available")
    md, hd, od = os.path.join(ROOT, "tests", "mock_engine"), os.path.join(ROOT, "bulletproofs_b200", "host"), os.path.join(ROOT, "oracle")
    objs = []
    for f in ("mock_bpmsm.c", "mock_stubs.c", "mock_ct_log.c"):
        o = os.path.join(tmp, f + ".o"); objs.append(o)
        subprocess.run(["gcc", "-O2", "-fPIC", "-c", "-o", o, os.path.join(md, f)], check=True)
    for f in ("bulletproofs.cpp", "r1cs.cpp", "mpc.cpp"):
        o = os.path.join(tmp, f + ".o"); objs.append(o)
        subprocess.run([_gxx(), "-O2", "-std=c++17", "-pthread", "-fPIC", "-DBP_HOST_REQUIRE_CT", "-c", "-o", o, os.path.join(hd, f)], check=True)
    so = os.path.join(tmp, "libroute.so")
    subprocess.run([_gxx(), "-shared", "-pthread", "-o", so] + objs + ["-L" + od, "-loracle", "-Wl,-rpath," + od, "-Wl,-Bsymbolic", "-Wl,-z,defs",
                    "-Wl,--wrap=bp_msm_indexed_batch", "-Wl,--wrap=bp_msm_batch"], check=True)
    return so


class Mock:
    def __init__(self, so):
        self.M = self.H = ctypes.CDLL(so)
        self.M.ct_log_entry.restype = ctypes.c_char_p
        self.M.ct_log_entry.argtypes = [ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t), ctypes.POINTER(ctypes.c_size_t), ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        self.M.ct_log_count.restype = ctypes.c_size_t
        self.ctx, self.gens = ctypes.c_void_p(), ctypes.c_void_p()
        assert self.M.bp_ctx_create(0, None, ctypes.byref(self.ctx)) == 0
        self.cap, self.parties = 64, 2
        assert self.M.bp_gens_create(self.ctx, ctypes.c_size_t(self.cap), ctypes.c_size_t(self.parties), ctypes.byref(self.gens)) == 0

    def transcript(self, label):
        st = ctypes.create_string_buffer(203)
        self.M.bp_transcript_new(label, ctypes.c_size_t(len(label)), st)
        return st

    def logged(self, fn):
        self.M.ct_log_reset()
        fn()
        calls = []
        for i in range(self.M.ct_log_count()):
            nt, nm = ctypes.c_size_t(), ctypes.c_size_t()
            self.M.ct_log_entry(i, ctypes.byref(nt), ctypes.byref(nm), None, None, None)
            idx, off, sc = (ctypes.c_uint32 * max(nt.value, 1))(), (ctypes.c_uint64 * (nm.value + 1))(), ctypes.create_string_buffer(32 * nt.value)
            name = self.M.ct_log_entry(i, ctypes.byref(nt), ctypes.byref(nm), idx, off, sc).decode()
            calls.append((name, list(idx)[:nt.value], list(off), [sc.raw[32 * k:32 * k + 32] for k in range(nt.value)]))
        self.M.ct_log_reset()
        return calls


@pytest.fixture(scope="module")
def mock(built, tmp_path_factory):
    return Mock(build_routing_lib(str(tmp_path_factory.mktemp("ct_routing"))))


def prove_multiple(mk, values, blindings):
    n, m = 8, len(values)
    def run():
        proof, V = ctypes.create_string_buffer(32 * (9 + 2 * 4)), ctypes.create_string_buffer(32 * m)
        rc = mk.H.bph_rangeproof_prove(mk.ctx, mk.gens, ctypes.c_size_t(mk.cap), ctypes.c_size_t(mk.parties), mk.transcript(b"ct routing"),
                                       (ctypes.c_uint64 * m)(*values), b"".join(le(b) for b in blindings), ctypes.c_size_t(m), ctypes.c_size_t(n), bytes(range(32)), proof, V)
        assert rc == 0
    return run


def mpc_party(mk, v, blinding):
    def run():
        sz, u64 = ctypes.c_size_t, ctypes.c_uint64
        y, z, x = le(12345), le(678), le(91011)
        assert mk.H.bph_mpc_party_bit_commitment(mk.ctx, mk.gens, sz(mk.cap), sz(mk.parties), u64(v), le(blinding), sz(8), sz(1), bytes(32), ctypes.create_string_buffer(96)) == 0
        assert mk.H.bph_mpc_party_poly_commitment(mk.ctx, mk.gens, sz(mk.cap), sz(mk.parties), u64(v), sz(8), sz(1), bytes(32), y, z, ctypes.create_string_buffer(64)) == 0
        assert mk.H.bph_mpc_party_proof_share(mk.ctx, mk.gens, sz(mk.cap), sz(mk.parties), u64(v), le(blinding), sz(8), sz(1), bytes(32), y, z, x, ctypes.create_string_buffer(32 * 19)) == 0
    return run


def r1cs_example(mk, values, blindings):
    def run():
        sz, u64 = ctypes.c_size_t, ctypes.c_uint64
        proof, n, V = ctypes.create_string_buffer(1 + 32 * 14 + 32 * 66), ctypes.c_size_t(), ctypes.create_string_buffer(32 * len(values))
        rc = mk.H.bph_r1cs_prove(mk.ctx, mk.gens, sz(mk.cap), sz(mk.parties), mk.transcript(b"R1CSExampleGadget"), ctypes.c_int(1), b"".join(le(v) for v in values),
                                 b"".join(le(b) for b in blindings), sz(len(values)), u64(9), u64(0), bytes(32), proof, ctypes.byref(n), V)
        assert rc == 0
    return run


@pytest.mark.parametrize("flow", ["prove_multiple", "mpc_party", "r1cs"])
def test_prover_secrets_reach_only_the_ct_entry_point(mock, flow):
    """Two runs with different values and blindings: every ct call has the same point indices and offsets in both, the
    commitments to secrets go to the ct entry point only, and the one variable-time indexed MSM is Q = w B (w a public challenge)."""
    rnd = random.Random(25)
    if flow == "prove_multiple":
        runs = [([3, 200], [rnd.randrange(l), rnd.randrange(l)]), ([255, 0], [rnd.randrange(l), rnd.randrange(l)])]
        make, n_ct = (lambda v, b: prove_multiple(mock, v, b)), 2             # [V_j, A, S], [T_1, T_2]
    elif flow == "mpc_party":
        runs = [(5, rnd.randrange(l)), (250, rnd.randrange(l))]
        make, n_ct = (lambda v, b: mpc_party(mock, v, b)), 5                  # V; A, S; then replayed for T_1/T_2 and the share
    else:
        runs = [([3, 4, 6, 1, 40], [rnd.randrange(l) for _ in range(5)]), ([7, 2, 5, 11, 99], [rnd.randrange(l) for _ in range(5)])]
        make, n_ct = (lambda v, b: r1cs_example(mock, v, b)), 3               # commitments; A_I1, A_O1, S1; T_1, T_3..T_6
    logs = [mock.logged(make(v, b)) for v, b in runs]
    shapes = []
    for (values, blindings), calls in zip(runs, logs):
        secrets = {le(x) for x in ([values] if isinstance(values, int) else values)} | {le(x) for x in ([blindings] if isinstance(blindings, int) else blindings)}
        ct = [c for c in calls if c[0] == CT]
        assert len(ct) >= n_ct, [c[0] for c in calls]
        assert {c[0] for c in calls} <= {CT, VT}, [c[0] for c in calls]
        assert secrets <= {s for c in ct for s in c[3]}, "a value or blinding never reached the ct entry point"
        for name, idx, off, sc in calls:
            if name == VT:
                assert idx == [1] and off == [0, 1], (idx, off)         # Q = w * B (slot 1)
                assert not (set(sc) & secrets)
        shapes.append([(c[1], c[2]) for c in ct])
    assert shapes[0] == shapes[1], "point indices or offsets of a constant-time call depend on the secrets"
