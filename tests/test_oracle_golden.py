"""CPU tier: the oracle against every fixed vector the reference holds for this path.

  - 16 golden proofs of /root/reference/tests/range_proof.rs:15-95 must verify (accept side),
  - the 8 golden commitments must be reproduced from their provenance (values 0..7, blindings from
    ChaChaRng::from_seed([24;32]), tests/range_proof.rs:108-113) — pins commit + compress + ChaCha + wide reduce,
  - Merlin known-answer (merlin crate's "test protocol" vector), generator/Pedersen constants (SURVEY.md §8c),
  - libsodium's independent ristretto255 (stored answers) for hash-to-group, point validity, addition and scalar multiplication.
"""
import json
import os
import random

import pytest

from oracle_binding import L_ORDER


def _blindings(orc, golden):
    return orc.random_scalars(bytes.fromhex(golden["commitment_blinding_rng_seed"]), 8)


def test_constants_and_generators(orc):
    B, Bb = orc.pedersen()
    assert B.hex() == "e2f2ae0a6abc4e71a884a961c500515f58e30b6aa582dd8db6a65945e08d2d76"
    assert Bb.hex() == "8c9240b456a9e6dc65c377a1048d745f94a08cdb7f44cbcd7b46f34048871134"
    g = orc.gens(64, 8)
    assert orc.gens_get(g, 0, 0, 0).hex() == "fc3b25801422672a6a8d3adb5d8457d4301fe92324b4fc56ae934c8713ddfe2d"
    assert orc.gens_get(g, 0, 0, 1).hex() == "ae817fdef62f713dd169dc8a26406f68be0bd3cd53652614636b0801567c4264"
    # capacity growth keeps the prefix (generators.rs:317-355 "resizing" test)
    g2 = orc.gens(16, 2)
    for which in (0, 1):
        for i in range(16):
            assert orc.gens_get(g2, which, 1, i) == orc.gens_get(g, which, 1, i)


def test_merlin_known_answer(orc):
    st = orc.transcript(b"test protocol")
    st = orc.transcript_append(st, b"some label", b"some data")
    _, ch = orc.transcript_challenge(st, b"challenge", 32)
    assert ch.hex() == "d5a21972d0d5fe320c0d263fac7fffb8145aa640af6e9bca177c03c7efcf0615"


def test_hashes_against_hashlib(orc):
    import hashlib
    for n in (0, 1, 71, 72, 73, 135, 136, 137, 500):
        d = bytes(range(256)) * 2
        d = d[:n]
        assert orc.sha3_512(d) == hashlib.sha3_512(d).digest()
        assert orc.shake256(d, 300) == hashlib.shake_256(d).digest(300)


def test_golden_proofs_verify(orc, golden):
    g = orc.gens(64, 8)
    vc = b"".join(bytes.fromhex(v) for v in golden["value_commitments"])
    t = orc.transcript(golden["transcript_label"].encode())
    for p in golden["proofs"]:
        proof = bytes.fromhex(p["proof"])
        assert len(proof) == orc.rangeproof_size(p["n"], p["m"])
        assert orc.rangeproof_verify(g, t, proof, vc[:32 * p["m"]], p["m"], p["n"]) == 0, (p["n"], p["m"])


def test_golden_proofs_reject_when_tampered(orc, golden):
    g = orc.gens(64, 8)
    vc = b"".join(bytes.fromhex(v) for v in golden["value_commitments"])
    t = orc.transcript(golden["transcript_label"].encode())
    rnd = random.Random(7)
    for p in golden["proofs"]:
        proof = bytearray(bytes.fromhex(p["proof"]))
        pos = rnd.randrange(len(proof))
        proof[pos] ^= 1 << rnd.randrange(8)
        assert orc.rangeproof_verify(g, t, bytes(proof), vc[:32 * p["m"]], p["m"], p["n"]) != 0
        # wrong commitment, wrong transcript label, wrong bitsize
        good = bytes.fromhex(p["proof"])
        wrong_vc = vc[32:32 * p["m"] + 32]
        assert orc.rangeproof_verify(g, t, good, wrong_vc, p["m"], p["n"]) != 0
        assert orc.rangeproof_verify(g, orc.transcript(b"other label"), good, vc[:32 * p["m"]], p["m"], p["n"]) != 0
        other_n = 8 if p["n"] != 8 else 16
        assert orc.rangeproof_verify(g, t, good, vc[:32 * p["m"]], p["m"], other_n) != 0


def test_golden_commitments_reproduced_by_prover(orc, golden):
    g = orc.gens(64, 8)
    bl = _blindings(orc, golden)
    t = orc.transcript(golden["transcript_label"].encode())
    for n, m in ((8, 1), (16, 2), (32, 4), (64, 8), (64, 1)):
        rc, proof, V = orc.rangeproof_prove(g, t, list(range(m)), bl[:32 * m], n, seed=bytes([n + m]) * 32)
        assert rc == 0
        assert V.hex() == "".join(golden["value_commitments"][:m])
        assert len(proof) == len(bytes.fromhex([p for p in golden["proofs"] if p["n"] == n and p["m"] == m][0]["proof"]))
        assert orc.rangeproof_verify(g, t, proof, V, m, n) == 0


def test_prover_is_deterministic_and_out_of_range_fails(orc, golden):
    g = orc.gens(64, 8)
    bl = _blindings(orc, golden)
    t = orc.transcript(b"AggregateRangeProofBenchmark")
    a = orc.rangeproof_prove(g, t, [123456789], bl[:32], 32, seed=bytes([24]) * 32)
    b = orc.rangeproof_prove(g, t, [123456789], bl[:32], 32, seed=bytes([24]) * 32)
    assert a == b and a[0] == 0 and len(a[1]) == 608
    rc, proof, V = orc.rangeproof_prove(g, t, [1 << 33], bl[:32], 32)
    assert rc == 0 and orc.rangeproof_verify(g, t, proof, V, 1, 32) != 0
    assert orc.rangeproof_prove(g, t, [1, 2, 3], bl[:96], 32)[0] == 5          # InvalidAggregation (m not a power of two)
    assert orc.rangeproof_prove(g, t, [1], bl[:32], 24)[0] == 3                # InvalidBitsize


def test_msm_algorithms_agree(orc):
    rnd = random.Random(3)
    pts = [orc.from_uniform(rnd.randbytes(64)) for _ in range(40)]
    for n in (1, 2, 5, 189, 190, 600, 900):        # Straus below 190 terms, Pippenger w=6/7/8 above
        sc = b"".join(rnd.randrange(L_ORDER).to_bytes(32, "little") for _ in range(n))
        pp = b"".join(rnd.choice(pts) for _ in range(n))
        assert orc.msm(sc, pp) == orc.msm(sc, pp, naive=True)
    assert orc.msm(b"", b"") == (0, bytes(32))
    assert orc.msm(L_ORDER.to_bytes(32, "little"), pts[0])[0] == 7     # non-canonical scalar
    assert orc.msm((1).to_bytes(32, "little"), b"\x01" + bytes(31))[0] == 6      # invalid point


def test_ipp_roundtrip(orc):
    """inner_product_proof.rs:433-534 (create -> verify), n in {1, 2, 4, 32, 64}."""
    rnd = random.Random(11)
    g = orc.gens(64, 1)
    Q = orc.from_uniform(orc.sha3_512(b"test point"))
    for n in (1, 2, 4, 32, 64):
        G = b"".join(orc.gens_get(g, 0, 0, i) for i in range(n))
        H = b"".join(orc.gens_get(g, 1, 0, i) for i in range(n))
        a = [rnd.randrange(L_ORDER) for _ in range(n)]
        b = [rnd.randrange(L_ORDER) for _ in range(n)]
        y_inv = rnd.randrange(1, L_ORDER)
        Gf = [1] * n
        Hf = [pow(y_inv, i, L_ORDER) for i in range(n)]
        c = sum(x * y for x, y in zip(a, b)) % L_ORDER
        enc = lambda xs: b"".join(x.to_bytes(32, "little") for x in xs)
        # P = <a, G> + <b', H> + c Q with b' = b * y^-i
        bprime = [x * h % L_ORDER for x, h in zip(b, Hf)]
        rc, P = orc.msm(enc(a) + enc(bprime) + enc([c]), G + H + Q)
        assert rc == 0
        t = orc.transcript(b"innerproducttest")
        rc, _, proof = orc.ipp_create(t, Q, enc(Gf), enc(Hf), G, H, enc(a), enc(b), n)
        assert rc == 0 and len(proof) == 32 * (2 * (n.bit_length() - 1) + 2)
        assert orc.ipp_verify(t, n, enc(Gf), enc(Hf), P, Q, G, H, proof) == 0
        bad = bytearray(proof); bad[-1] ^= 1
        assert orc.ipp_verify(t, n, enc(Gf), enc(Hf), P, Q, G, H, bytes(bad)) != 0


def test_group_against_libsodium(orc):
    """libsodium's answers, stored by tests/golden/make_libsodium_golden.py"""
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ristretto255_libsodium.json")) as f:
        sod = json.load(f)
    assert (len(sod["from_hash"]), len(sod["add"]), len(sod["scalarmult"]), len(sod["is_valid_point"])) == (50, 50, 50, 300)
    pts = []
    for h, want in sod["from_hash"]:
        got = orc.from_uniform(bytes.fromhex(h))
        assert got.hex() == want and orc.point_is_valid(got) == 1
        pts.append(got)
    for i, j, want in sod["add"]:
        assert orc.point_add(pts[i], pts[j]).hex() == want
    for s, i, want in sod["scalarmult"]:
        assert orc.msm(bytes.fromhex(s), pts[i]) == (0, bytes.fromhex(want))
    for s, want in sod["is_valid_point"]:
        assert orc.point_is_valid(bytes.fromhex(s)) == want


@pytest.mark.parametrize("backend", ["avx2", "ifma"])
def test_vector_backends_pinned_like_the_serial_one(orc, golden, backend):
    """The 4-way vector field backends of the oracle's MSM (oracle/vec4_avx2.h: the reference's default `avx2_backend`,
    Cargo.toml:41-42; oracle/vec4_ifma.h: README.md:82-84) against the same pins as the serial u64 code: field / point
    self-test vs the serial code, MSM results identical at Straus and Pippenger sizes, all 16 golden proofs accept,
    tampered ones reject, the prover's bytes do not depend on the backend."""
    if orc.set_backend(backend) != 0:
        orc.set_backend("u64")
        pytest.skip(f"this CPU has no {backend}")
    try:
        rnd = random.Random(11)
        pts = [orc.from_uniform(rnd.randbytes(64)) for _ in range(48)]
        edge = [2**255 - 20, 2**255 - 21, 0, 1, 2**255 - 1, 2**254, 2**51 - 1, 19]
        for t in range(100):
            r8 = b"".join(x.to_bytes(32, "little") for x in edge) if t == 0 else b"".join(rnd.getrandbits(255).to_bytes(32, "little") for _ in range(8))
            assert orc.vec_selftest(backend, b"".join(rnd.choice(pts) for _ in range(4)), r8) == 0
        for n in (1, 2, 3, 17, 147, 189, 190, 499, 500, 800, 2090):
            sc = b"".join(rnd.randrange(L_ORDER).to_bytes(32, "little") for _ in range(n)); pp = b"".join(rnd.choice(pts) for _ in range(n))
            got = orc.msm(sc, pp)
            orc.set_backend("u64"); want = orc.msm(sc, pp); orc.set_backend(backend)
            assert got == want, n
        special = b"".join(x.to_bytes(32, "little") for x in (0, 1, L_ORDER - 1, 2**252, 2**128, 5)); pp = b"".join(pts[:6])
        got = orc.msm(special, pp); orc.set_backend("u64"); assert got == orc.msm(special, pp); orc.set_backend(backend)
        assert orc.msm((7).to_bytes(32, "little") + (L_ORDER - 7).to_bytes(32, "little"), pts[0] * 2) == (0, bytes(32))
        g = orc.gens(64, 8)
        vc = b"".join(bytes.fromhex(v) for v in golden["value_commitments"])
        t = orc.transcript(golden["transcript_label"].encode())
        for p in golden["proofs"]:
            proof = bytes.fromhex(p["proof"])
            assert orc.rangeproof_verify(g, t, proof, vc[:32 * p["m"]], p["m"], p["n"]) == 0, (backend, p["n"], p["m"])
            bad = bytearray(proof); bad[rnd.randrange(len(bad))] ^= 1 << rnd.randrange(8)
            assert orc.rangeproof_verify(g, t, bytes(bad), vc[:32 * p["m"]], p["m"], p["n"]) != 0
        rc, proof_v, V_v = orc.rangeproof_prove(g, t, [3, 250], (5).to_bytes(32, "little") + (6).to_bytes(32, "little"), 8)
        orc.set_backend("u64")
        assert (rc, proof_v, V_v) == orc.rangeproof_prove(g, t, [3, 250], (5).to_bytes(32, "little") + (6).to_bytes(32, "little"), 8) and rc == 0
        assert "u64" in orc.backend_name()
    finally:
        orc.set_backend("u64")
