"""Stores libsodium's ristretto255 answers as a JSON fixture, so that the oracle's group arithmetic is checked against an
independent implementation without libsodium being installed.

Inputs are drawn from random.Random(5): 50 hash-to-group inputs, 50 additions and scalar multiplications of the resulting
points, 300 random 32-byte strings for the validity check.  tests/test_oracle_golden.py::test_group_against_libsodium checks
the oracle against every stored answer.
    python tests/golden/make_libsodium_golden.py /path/to/libsodium.so
"""
import ctypes
import json
import pathlib
import random
import sys

L_ORDER = 2**252 + 27742317777372353535851937790883648493

sod = ctypes.CDLL(sys.argv[1])
sod.sodium_version_string.restype = ctypes.c_char_p
rnd = random.Random(5)
o = ctypes.create_string_buffer(32)
from_hash, pts = [], []
for _ in range(50):
    h = rnd.randbytes(64)
    assert sod.crypto_core_ristretto255_from_hash(o, h) == 0 and sod.crypto_core_ristretto255_is_valid_point(o.raw) == 1
    from_hash.append([h.hex(), o.raw.hex()])
    pts.append(o.raw)
add, mul = [], []
for _ in range(50):
    a, b = rnd.choice(pts), rnd.choice(pts)
    assert sod.crypto_core_ristretto255_add(o, a, b) == 0
    add.append([pts.index(a), pts.index(b), o.raw.hex()])
    s = rnd.randrange(1, L_ORDER).to_bytes(32, "little")
    assert sod.crypto_scalarmult_ristretto255(o, s, a) == 0
    mul.append([s.hex(), pts.index(a), o.raw.hex()])
valid = []
for _ in range(300):
    s = rnd.randbytes(32)
    valid.append([s.hex(), sod.crypto_core_ristretto255_is_valid_point(s)])
out = {"source": f"libsodium {sod.sodium_version_string().decode()}: crypto_core_ristretto255_{{from_hash,add,is_valid_point}}, "
                 "crypto_scalarmult_ristretto255",
       "from_hash": from_hash,             # [64-byte input, point]
       "add": add,                         # [index of a, index of b, a + b]; indices into from_hash
       "scalarmult": mul,                  # [scalar, index of the point, scalar * point]
       "is_valid_point": valid}            # [32 bytes, 1 if they encode a point]
pathlib.Path(__file__).with_name("ristretto255_libsodium.json").write_text(json.dumps(out, indent=0) + "\n")
print("wrote", len(from_hash), len(add), len(mul), len(valid))
