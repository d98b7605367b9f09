"""bulletproofs_b200 — Python harness over the C ABI of the B200-native Bulletproofs MSM engine.

Everything here is a thin ctypes view of include/bpmsm.h (libbpmsm.so, hand-written sm_100a CUDA).
There is no CPU path: importing works without a GPU (so the symbol table can be checked), but every
compute call needs a B200 and raises otherwise.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbpmsm.so")

TRANSCRIPT_BYTES = 203
OK, ERR_INVALID_POINT, ERR_LENGTH_MISMATCH, ERR_NONCANONICAL_SCALAR, ERR_CUDA, ERR_INVALID_ARGUMENT = range(6)
PROOF_OK, PROOF_VERIFICATION_ERROR, PROOF_FORMAT_ERROR, PROOF_INVALID_BITSIZE, PROOF_INVALID_GENERATORS_LENGTH, PROOF_INVALID_AGGREGATION = range(6)

_c = ctypes
_vp, _sz, _u8p, _int = _c.c_void_p, _c.c_size_t, _c.c_char_p, _c.c_int

# every symbol include/bpmsm.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "bp_ctx_create": (_int, [_int, _vp, _c.POINTER(_vp)]),
    "bp_ctx_destroy": (None, [_vp]),
    "bp_last_error": (_c.c_char_p, [_vp]),
    "bp_ctx_launch_count": (_c.c_uint64, [_vp]),
    "bp_ctx_synchronize": (_int, [_vp]),
    "bp_ctx_set_msm_window": (_int, [_vp, _int]),
    "bp_decompress_check_batch": (_int, [_vp, _u8p, _sz, _u8p]),
    "bp_from_uniform_bytes_batch": (_int, [_vp, _u8p, _sz, _u8p]),
    "bp_decompress_batch": (_int, [_vp, _u8p, _sz, _u8p, _u8p]),
    "bp_compress_batch": (_int, [_vp, _u8p, _sz, _u8p]),
    "bp_points_create": (_int, [_vp, _vp, _sz, _c.POINTER(_vp)]),
    "bp_points_create_device": (_int, [_vp, _vp, _sz, _c.POINTER(_vp)]),
    "bp_points_destroy": (None, [_vp]),
    "bp_points_count": (_sz, [_vp]),
    "bp_msm_points_device": (_int, [_vp, _vp, _vp, _sz, _sz, _vp, _vp]),
    "bp_msm_points": (_int, [_vp, _vp, _vp, _sz, _sz, _vp, _vp]),
    "bp_msm": (_int, [_vp, _u8p, _u8p, _sz, _u8p]),
    "bp_msm_batch": (_int, [_vp, _u8p, _u8p, _c.POINTER(_c.c_uint64), _sz, _u8p, _u8p]),
    "bp_msm_batch_device": (_int, [_vp, _vp, _vp, _vp, _sz, _sz, _vp, _vp]),
    "bp_msm_indexed_batch": (_int, [_vp, _vp, _u8p, _c.POINTER(_c.c_uint32), _u8p, _sz, _c.POINTER(_c.c_uint64), _sz, _u8p, _u8p]),
    "bp_ipp_begin_points": (_int, [_vp, _u8p, _u8p, _sz, _u8p, _c.POINTER(_vp)]),
    "bp_ipp_lr": (_int, [_vp, _sz, _u8p, _u8p, _u8p, _u8p]),
    "bp_ipp_fold": (_int, [_vp, _sz, _u8p, _u8p, _u8p, _u8p, _int]),
    "bp_ipp_end": (None, [_vp]),
    "bp_ippx_begin": (_int, [_vp, _vp, _sz, _sz, _sz, _u8p, _u8p, _u8p, _u8p, _u8p, _c.POINTER(_vp)]),
    "bp_ippx_begin_points": (_int, [_vp, _u8p, _u8p, _sz, _sz, _u8p, _u8p, _u8p, _u8p, _u8p, _c.POINTER(_vp)]),
    "bp_ippx_current_len": (_sz, [_vp]),
    "bp_ippx_round": (_int, [_vp, _u8p]),
    "bp_ippx_fold": (_int, [_vp, _u8p, _u8p]),
    "bp_ippx_finish": (_int, [_vp, _u8p]),
    "bp_ippx_end": (None, [_vp]),
    "bp_gens_create": (_int, [_vp, _sz, _sz, _c.POINTER(_vp)]),
    "bp_gens_create_empty": (_int, [_vp, _sz, _sz, _c.POINTER(_vp)]),
    "bp_gens_destroy": (None, [_vp]),
    "bp_gens_get": (_int, [_vp, _int, _sz, _sz, _u8p]),
    "bp_gens_device_table": (_int, [_vp, _c.POINTER(_vp), _c.POINTER(_sz)]),
    "bp_rangeproof_verify_batch": (_int, [_vp, _vp, _u8p, _u8p, _sz, _u8p, _sz, _sz, _sz, _u8p, _u8p]),
    "bp_rangeproof_verify_begin": (_int, [_vp, _vp, _u8p, _vp, _sz, _vp, _sz, _sz, _sz, _u8p]),
    "bp_rangeproof_verify_finish": (_int, [_vp, _u8p]),
    "bp_rangeproof_verify_batch_device": (_int, [_vp, _vp, _u8p, _vp, _sz, _vp, _sz, _sz, _sz, _u8p, _vp, _vp]),
    "bp_rangeproof_verify_group_begin": (_int, [_vp, _vp, _u8p, _vp, _sz, _vp, _sz, _sz, _sz, _sz, _u8p]),
    "bp_rangeproof_verify_group_finish": (_int, [_vp, _u8p, _u8p]),
    "bp_rangeproof_verify_group_device": (_int, [_vp, _vp, _u8p, _vp, _sz, _vp, _sz, _sz, _sz, _sz, _u8p, _vp, _vp]),
    "bp_rangeproof_verify_reserve": (_int, [_vp, _vp, _sz, _sz, _sz, _sz]),
    "bp_gens_table_export": (_int, [_vp, _vp]),
    "bp_gens_table_import": (_int, [_vp, _vp]),
    "bp_prof_enable": (_int, [_vp, _int]),
    "bp_prof_kernel_count": (_int, []),
    "bp_prof_kernel_name": (_c.c_char_p, [_int]),
    "bp_prof_report": (_int, [_vp, _c.POINTER(_c.c_double), _c.POINTER(_c.c_uint64)]),
    "bp_prof_timeline": (_int, [_vp, _vp, _c.POINTER(_c.c_int), _c.POINTER(_c.c_double), _c.POINTER(_c.c_double), _c.c_size_t, _c.POINTER(_c.c_size_t)]),
    "bp_transcript_new": (None, [_u8p, _sz, _u8p]),
    "bp_transcript_append_message": (None, [_u8p, _u8p, _u8p, _sz]),
    "bp_transcript_append_u64": (None, [_u8p, _u8p, _c.c_uint64]),
    "bp_transcript_challenge_bytes": (None, [_u8p, _u8p, _u8p, _sz]),
    "bp_debug_fe_op": (_int, [_vp, _int, _u8p, _u8p, _sz, _u8p]),
}


# the constant-time entry points, declared in include/bpmsm_ct.h; bound on first use by ct_lib()
CT_SYMBOLS = {
    "bp_msm_indexed_batch_ct": (_int, [_vp, _vp, _u8p, _c.POINTER(_c.c_uint32), _c.POINTER(_c.c_uint64), _sz, _u8p, _u8p]),
}


class BpError(RuntimeError):
    def __init__(self, code, msg=""):
        super().__init__(f"bpmsm error {code}: {msg}")
        self.code = code


_lib = None


def lib():
    """Load libbpmsm.so (loudly: a missing CUDA extension is an error, never a fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a)")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)          # AttributeError if the library does not export a declared symbol
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


_ct_bound = False


def ct_lib():
    """libbpmsm.so with the constant-time entry points of include/bpmsm_ct.h bound as well (AttributeError if one is missing)."""
    global _ct_bound
    L = lib()
    if not _ct_bound:
        for name, (res, args) in CT_SYMBOLS.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _ct_bound = True
    return L


HOST_LIB_PATH = os.path.join(_HERE, "libbulletproofs_host.so")
_hlib = None


def host_lib():
    """C shim of the C++ mirror of the reference API (bulletproofs_b200/host): prover-side entry points."""
    global _hlib
    if _hlib is None:
        lib()
        if not os.path.exists(HOST_LIB_PATH):
            raise ImportError(f"{HOST_LIB_PATH} is missing: run build()")
        H = ctypes.CDLL(HOST_LIB_PATH)
        H.bph_rangeproof_prove.restype = _int
        H.bph_rangeproof_prove.argtypes = [_vp, _vp, _sz, _sz, _u8p, _c.POINTER(_c.c_uint64), _u8p, _sz, _sz, _u8p, _u8p, _u8p]
        H.bph_rangeproof_prove_many.restype = _int
        H.bph_rangeproof_prove_many.argtypes = [_vp, _vp, _sz, _sz, _u8p, _c.POINTER(_c.c_uint64), _u8p, _sz, _sz, _sz, _u8p, _u8p, _sz, _u8p, _u8p]
        H.bph_rangeproof_verify.restype = _int
        H.bph_rangeproof_verify.argtypes = [_vp, _vp, _sz, _sz, _u8p, _u8p, _sz, _u8p, _sz, _sz]
        H.bph_ipp_create.restype = _int
        H.bph_ipp_create.argtypes = [_vp, _u8p, _u8p, _u8p, _u8p, _u8p, _u8p, _u8p, _u8p, _sz, _u8p]
        H.bph_ipp_verify.restype = _int
        H.bph_ipp_verify.argtypes = [_vp, _u8p, _sz, _u8p, _u8p, _u8p, _u8p, _u8p, _u8p, _u8p, _sz]
        H.bph_linear_create.restype = _int
        H.bph_linear_create.argtypes = [_vp, _u8p, _u8p, _u8p, _u8p, _u8p, _u8p, _u8p, _u8p, _u8p, _sz, _u8p]
        H.bph_linear_verify.restype = _int
        H.bph_linear_verify.argtypes = [_vp, _u8p, _u8p, _sz, _u8p, _u8p, _u8p, _u8p, _u8p, _sz]
        H.bph_r1cs_prove.restype = _int
        H.bph_r1cs_prove.argtypes = [_vp, _vp, _sz, _sz, _u8p, _int, _u8p, _u8p, _sz, _c.c_uint64, _c.c_uint64, _u8p, _u8p, _c.POINTER(_sz), _u8p]
        H.bph_r1cs_verify.restype = _int
        H.bph_r1cs_verify.argtypes = [_vp, _vp, _sz, _sz, _u8p, _int, _u8p, _sz, _c.c_uint64, _u8p, _sz, _u8p]
        u64 = _c.c_uint64
        for name, args in (("bph_mpc_party_bit_commitment", [_vp, _vp, _sz, _sz, u64, _u8p, _sz, _sz, _u8p, _u8p]),
                           ("bph_mpc_party_poly_commitment", [_vp, _vp, _sz, _sz, u64, _sz, _sz, _u8p, _u8p, _u8p, _u8p]),
                           ("bph_mpc_party_proof_share", [_vp, _vp, _sz, _sz, u64, _u8p, _sz, _sz, _u8p, _u8p, _u8p, _u8p, _u8p]),
                           ("bph_mpc_audit_share", [_vp, _vp, _sz, _sz, _sz, _sz, _u8p, _u8p, _u8p, _u8p, _u8p, _u8p]),
                           ("bph_mpc_dealer_run", [_vp, _vp, _sz, _sz, _u8p, _sz, _sz, _u8p, _u8p, _u8p, _int, _u8p, _u8p, _u8p])):
            getattr(H, name).restype = _int
            getattr(H, name).argtypes = args
        _hlib = H
    return _hlib


GADGET_SHUFFLE, GADGET_EXAMPLE, GADGET_RANGE = 0, 1, 2


def r1cs_prove(ctx, gens, transcript, gadget: int, values, blindings: bytes, param: int = 0, aux: int = 0, ext_seed: bytes = bytes(32)):
    """r1cs::Prover::{new, commit.., prove} with one of the reference's gadgets (shuffle: values = inputs then outputs;
    example: a1,a2,b1,b2,c1 with param = c2; range: one value with param = n bits, aux = the value).  Returns
    (status, R1CSProof::to_bytes(), commitments); ext_seed seeds the external RNG that finalises the TranscriptRng."""
    m = len(values)
    vals = b"".join(int(v).to_bytes(32, "little") for v in values)
    proof = ctypes.create_string_buffer(1 + 32 * 14 + 32 * (2 * 32 + 2))
    n = _sz()
    V = ctypes.create_string_buffer(32 * max(m, 1))
    rc = host_lib().bph_r1cs_prove(ctx._h, gens._h, gens.gens_capacity, gens.party_capacity, transcript.state, gadget, vals, blindings, m, param, aux, ext_seed, proof, ctypes.byref(n), V)
    if rc < 0:
        raise BpError(rc, lib().bp_last_error(ctx._h).decode())
    return rc, proof.raw[:n.value], V.raw[:32 * m]


def r1cs_verify(ctx, gens, transcript, gadget: int, commitments: bytes, proof: bytes, param: int = 0, ext_seed: bytes = bytes(32)) -> int:
    rc = host_lib().bph_r1cs_verify(ctx._h, gens._h, gens.gens_capacity, gens.party_capacity, transcript.to_bytes(), gadget, commitments, len(commitments) // 32, param, proof, len(proof), ext_seed)
    if rc < 0:
        raise BpError(rc, lib().bp_last_error(ctx._h).decode())
    return rc


class Transcript:
    """merlin::Transcript on the 203-byte wire state (host helper of the C ABI)."""

    def __init__(self, label: bytes = None, state: bytes = None):
        self.state = ctypes.create_string_buffer(TRANSCRIPT_BYTES)
        if state is not None:
            self.state.raw = bytes(state)
        else:
            lib().bp_transcript_new(label, len(label), self.state)

    def clone(self):
        return Transcript(state=self.state.raw)

    def append_message(self, label: bytes, msg: bytes):
        lib().bp_transcript_append_message(self.state, label, msg, len(msg))

    def append_u64(self, label: bytes, x: int):
        lib().bp_transcript_append_u64(self.state, label, x)

    def challenge_bytes(self, label: bytes, n: int) -> bytes:
        out = ctypes.create_string_buffer(n)
        lib().bp_transcript_challenge_bytes(self.state, label, out, n)
        return out.raw

    def to_bytes(self) -> bytes:
        return self.state.raw


class Context:
    """One device + one CUDA stream (bp_ctx)."""

    def __init__(self, device: int = 0, stream: int = None):
        self._h = _vp()
        rc = lib().bp_ctx_create(device, _vp(stream) if stream else None, ctypes.byref(self._h))
        if rc != OK:
            raise BpError(rc, "bp_ctx_create failed: no usable sm_100 CUDA device (there is no CPU fallback)")
        self.device = device

    def close(self):
        if self._h:
            lib().bp_ctx_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != OK:
            raise BpError(rc, lib().bp_last_error(self._h).decode())

    @property
    def launches(self) -> int:
        return lib().bp_ctx_launch_count(self._h)

    def synchronize(self):
        self._check(lib().bp_ctx_synchronize(self._h))

    def set_msm_window(self, bits: int):
        """Pippenger window of the generic MSM entry points: 0 = by size (default), 2..18 = fixed"""
        self._check(lib().bp_ctx_set_msm_window(self._h, bits))

    def prof_enable(self, on=True):
        self._check(lib().bp_prof_enable(self._h, 1 if on else 0))

    def prof_report(self):
        """{kernel name: (total ms, launches)} from CUDA events since the last report (synchronises)."""
        n = lib().bp_prof_kernel_count()
        ms, cnt = (ctypes.c_double * n)(), (ctypes.c_uint64 * n)()
        self._check(lib().bp_prof_report(self._h, ms, cnt))
        return {lib().bp_prof_kernel_name(i).decode(): (ms[i], cnt[i]) for i in range(n) if cnt[i]}

    # ---- group primitives
    def prof_timeline(self, ref: "Context", cap: int = 65536):
        """[(kernel name, start ms, end ms)] of every launch recorded since prof_enable, relative to ref's first record."""
        ids = (ctypes.c_int * cap)(); a = (ctypes.c_double * cap)(); b = (ctypes.c_double * cap)(); n = ctypes.c_size_t(0)
        self._check(lib().bp_prof_timeline(self._h, ref._h, ids, a, b, cap, ctypes.byref(n)))
        return [(lib().bp_prof_kernel_name(ids[i]).decode(), a[i], b[i]) for i in range(n.value)]

    def decompress_check(self, points: bytes):
        n = len(points) // 32
        ok = ctypes.create_string_buffer(max(n, 1))
        self._check(lib().bp_decompress_check_batch(self._h, points, n, ok))
        return list(ok.raw[:n])

    def from_uniform_bytes(self, uniform: bytes) -> bytes:
        n = len(uniform) // 64
        out = ctypes.create_string_buffer(32 * max(n, 1))
        self._check(lib().bp_from_uniform_bytes_batch(self._h, uniform, n, out))
        return out.raw[:32 * n]

    def decompress(self, points: bytes):
        """CompressedRistretto::decompress for n points -> (list of 128-byte X|Y|Z|T values, ok flags)"""
        n = len(points) // 32
        out = ctypes.create_string_buffer(128 * max(n, 1)); ok = ctypes.create_string_buffer(max(n, 1))
        self._check(lib().bp_decompress_batch(self._h, points, n, out, ok))
        return [out.raw[128 * i:128 * i + 128] for i in range(n)], list(ok.raw[:n])

    def compress(self, xyzt: bytes) -> bytes:
        n = len(xyzt) // 128
        out = ctypes.create_string_buffer(32 * max(n, 1))
        self._check(lib().bp_compress_batch(self._h, xyzt, n, out))
        return out.raw[:32 * n]

    # ---- MSM
    def msm(self, scalars: bytes, points: bytes):
        """RistrettoPoint::vartime_multiscalar_mul; returns (status, 32-byte compressed result)."""
        if len(scalars) != len(points) or len(scalars) % 32:
            raise BpError(ERR_LENGTH_MISMATCH, "scalars/points length mismatch")
        out = ctypes.create_string_buffer(32)
        rc = lib().bp_msm(self._h, scalars, points, len(scalars) // 32, out)
        if rc in (ERR_CUDA, ERR_INVALID_ARGUMENT):
            self._check(rc)
        return rc, out.raw

    def msm_batch(self, scalars: bytes, points: bytes, offsets):
        n_msm = len(offsets) - 1
        offs = (ctypes.c_uint64 * (n_msm + 1))(*offsets)
        outs = ctypes.create_string_buffer(32 * n_msm)
        status = ctypes.create_string_buffer(n_msm)
        self._check(lib().bp_msm_batch(self._h, scalars, points, offs, n_msm, outs, status))
        return list(status.raw), [outs.raw[32 * i:32 * i + 32] for i in range(n_msm)]

    def debug_fe_op(self, op: int, a: bytes, b: bytes) -> bytes:
        n = len(a) // 32
        out = ctypes.create_string_buffer(32 * n)
        self._check(lib().bp_debug_fe_op(self._h, op, a, b, n, out))
        return out.raw


class PointSet:
    """n points decompressed once and resident on the device (bp_points): bases of repeated MSMs."""

    def __init__(self, ctx: Context, points=None, n: int = None, device_ptr: int = None):
        self.ctx, self._h = ctx, _vp()
        if device_ptr is not None:
            ctx._check(lib().bp_points_create_device(ctx._h, device_ptr, n, ctypes.byref(self._h)))
        else:
            n = len(points) // 32 if n is None else n
            buf = ctypes.create_string_buffer(bytes(points), 32 * n) if isinstance(points, (bytes, bytearray)) else None
            ctx._check(lib().bp_points_create(ctx._h, ctypes.addressof(buf) if buf is not None else points, n, ctypes.byref(self._h)))
        self.n = n

    def msm(self, scalars: bytes, n_msm: int, terms: int):
        """n_msm MSMs of `terms` terms over the first `terms` points; returns (status list, list of 32-byte results)"""
        outs = ctypes.create_string_buffer(32 * n_msm); st = ctypes.create_string_buffer(n_msm)
        buf = ctypes.create_string_buffer(bytes(scalars), 32 * n_msm * terms)
        self.ctx._check(lib().bp_msm_points(self.ctx._h, self._h, ctypes.addressof(buf), n_msm, terms, ctypes.addressof(outs), ctypes.addressof(st)))
        return list(st.raw), [outs.raw[32 * i:32 * i + 32] for i in range(n_msm)]

    def msm_device(self, d_scalars: int, n_msm: int, terms: int, d_outs: int, d_status: int = None):
        self.ctx._check(lib().bp_msm_points_device(self.ctx._h, self._h, d_scalars, n_msm, terms, d_outs, d_status))

    def close(self):
        if self._h:
            lib().bp_points_destroy(self._h)
            self._h = _vp()


class Gens:
    """BulletproofGens::new(gens_capacity, party_capacity) + PedersenGens::default(), resident on the device."""

    def __init__(self, ctx: Context, gens_capacity: int, party_capacity: int, empty: bool = False):
        self.ctx, self.gens_capacity, self.party_capacity = ctx, gens_capacity, party_capacity
        self._h = _vp()
        fn = lib().bp_gens_create_empty if empty else lib().bp_gens_create
        ctx._check(fn(ctx._h, gens_capacity, party_capacity, ctypes.byref(self._h)))

    def get(self, which: int, party: int = 0, index: int = 0) -> bytes:
        out = ctypes.create_string_buffer(32)
        self.ctx._check(lib().bp_gens_get(self._h, which, party, index, out))
        return out.raw

    def G(self, party, index):
        return self.get(0, party, index)

    def H(self, party, index):
        return self.get(1, party, index)

    @property
    def B(self):
        return self.get(2)

    @property
    def B_blinding(self):
        return self.get(3)

    def msm_indexed(self, scalars: bytes, point_idx, offsets, dyn_points: bytes = b"", constant_time: bool = False):
        """MSMs over table slots (bp_msm_indexed_batch): MSM j = sum of scalars[t] * slot point_idx[t] for t in offsets[j] .. offsets[j+1]-1;
        slot layout: 0 = B_blinding, 1 = B, 2 + party*cap + i = G[party][i], 2 + (parties + party)*cap + i = H[party][i].
        constant_time=True runs bp_msm_indexed_batch_ct (secret scalars; table slots only, no dyn_points).
        Returns (status list, list of 32-byte results)."""
        n_msm, T = len(offsets) - 1, len(point_idx)
        idx = (ctypes.c_uint32 * max(T, 1))(*point_idx)
        offs = (ctypes.c_uint64 * (n_msm + 1))(*offsets)
        outs, st = ctypes.create_string_buffer(32 * max(n_msm, 1)), ctypes.create_string_buffer(max(n_msm, 1))
        if constant_time:
            if dyn_points:
                raise BpError(ERR_INVALID_ARGUMENT, "the constant-time MSM takes table slots only")
            rc = ct_lib().bp_msm_indexed_batch_ct(self.ctx._h, self._h, scalars, idx, offs, n_msm, outs, st)
        else:
            rc = lib().bp_msm_indexed_batch(self.ctx._h, self._h, scalars, idx, dyn_points or None, len(dyn_points) // 32, offs, n_msm, outs, st)
        self.ctx._check(rc)
        return list(st.raw[:n_msm]), [outs.raw[32 * i:32 * i + 32] for i in range(n_msm)]

    def slot_G(self, party: int, index: int) -> int:
        return 2 + party * self.gens_capacity + index

    def slot_H(self, party: int, index: int) -> int:
        return 2 + (self.party_capacity + party) * self.gens_capacity + index

    def table_export(self, d_dst: int):
        self.ctx._check(lib().bp_gens_table_export(self._h, d_dst))

    def table_import(self, d_src: int):
        self.ctx._check(lib().bp_gens_table_import(self._h, d_src))

    def device_table(self):
        p, n = _vp(), _sz()
        self.ctx._check(lib().bp_gens_device_table(self._h, ctypes.byref(p), ctypes.byref(n)))
        return p.value, n.value

    def close(self):
        if self._h:
            lib().bp_gens_destroy(self._h)
            self._h = _vp()


class BatchVerifier:
    """Pipelined form of the batch verifier over raw buffers (bench.py): `n_batches` independent batches of `count` proofs per
    launch group.  The constructor reserves the geometry on the context (arenas sized, launch sequence captured as a CUDA graph,
    one warm pass) so that no later call allocates.  `begin` queues the H2D copies, the graph and the verdict D2H on the
    context's stream, `finish` synchronises and returns (verdict codes, per-batch accept flags)."""

    def __init__(self, ctx: Context, gens: Gens, transcript: Transcript, n: int, m: int, count: int, n_batches: int = 1, reserve: bool = True):
        self.ctx, self.gens, self.n, self.m, self.count, self.n_batches = ctx, gens, n, m, count, n_batches
        self.t = transcript.to_bytes()
        self.proof_len = rangeproof_size(n, m)
        self._verdicts = ctypes.create_string_buffer(count * n_batches)
        self._batch_ok = ctypes.create_string_buffer(n_batches)
        self.busy = False
        if reserve:
            ctx._check(lib().bp_rangeproof_verify_reserve(ctx._h, gens._h, n, m, count, n_batches))

    def begin(self, proofs_ptr: int, commitments_ptr: int, seed: bytes = None):
        """proofs_ptr / commitments_ptr: host addresses (pinned memory for truly asynchronous copies)."""
        self.ctx._check(lib().bp_rangeproof_verify_group_begin(self.ctx._h, self.gens._h, self.t, proofs_ptr, self.proof_len, commitments_ptr,
                                                               self.n, self.m, self.count, self.n_batches, seed))
        self.busy = True

    def finish(self):
        self.ctx._check(lib().bp_rangeproof_verify_group_finish(self.ctx._h, self._verdicts, self._batch_ok))
        self.busy = False
        self.batch_ok = list(self._batch_ok.raw)
        return self._verdicts.raw

    def run_device(self, d_proofs: int, d_commitments: int, d_verdicts_u32: int, h_batch_ok_pinned: int = None, seed: bytes = None):
        """device-resident inputs; nothing is synchronised (verdicts stay on the device)."""
        self.ctx._check(lib().bp_rangeproof_verify_group_device(self.ctx._h, self.gens._h, self.t, d_proofs, self.proof_len, d_commitments,
                                                                self.n, self.m, self.count, self.n_batches, seed, d_verdicts_u32, h_batch_ok_pinned))


def prove_multiple(ctx: Context, gens: Gens, transcript: Transcript, values, blindings: bytes, n: int, rng_seed: bytes):
    """RangeProof::prove_multiple_with_rng with rng = ChaChaRng::from_seed(rng_seed) on the GPU-backed path.
    Returns (status, proof bytes, commitments bytes); the transcript is advanced like the reference's &mut Transcript."""
    m = len(values)
    vals = (ctypes.c_uint64 * m)(*values)
    proof = ctypes.create_string_buffer(rangeproof_size(n, m) if m and (n * m) & (n * m - 1) == 0 else 32 * 64)
    V = ctypes.create_string_buffer(32 * max(m, 1))
    rc = host_lib().bph_rangeproof_prove(ctx._h, gens._h, gens.gens_capacity, gens.party_capacity, transcript.state, vals, blindings, m, n, rng_seed, proof, V)
    if rc < 0:
        raise BpError(rc, lib().bp_last_error(ctx._h).decode())
    return rc, proof.raw, V.raw


def prove_many(ctx: Context, gens: Gens, transcript: Transcript, values, blindings: bytes, n: int, m: int, rng_seeds: bytes):
    """`count` = len(values) // m independent aggregated proofs with every group operation batched across the proofs (one device call per
    prover phase, one inner-product session for all).  Proof p uses values[p*m:(p+1)*m] and ChaChaRng::from_seed(rng_seeds[32p:32p+32]);
    every transcript starts from `transcript`.  Returns (status list, proofs bytes, commitments bytes) -- the same bytes as `count` prove_multiple calls."""
    count = len(values) // m
    vals = (ctypes.c_uint64 * len(values))(*values)
    plen = rangeproof_size(n, m)
    proofs = ctypes.create_string_buffer(plen * count); V = ctypes.create_string_buffer(32 * m * count); st = ctypes.create_string_buffer(count)
    rc = host_lib().bph_rangeproof_prove_many(ctx._h, gens._h, gens.gens_capacity, gens.party_capacity, transcript.to_bytes(), vals, blindings, m, n, count, rng_seeds, proofs, plen, V, st)
    if rc < 0:
        raise BpError(rc, lib().bp_last_error(ctx._h).decode())
    return list(st.raw), proofs.raw, V.raw


def verify_multiple(ctx: Context, gens: Gens, transcript: Transcript, proof: bytes, commitments: bytes, n: int) -> int:
    """RangeProof::from_bytes + verify_multiple through the C++ mirror; returns the ProofError code (0 = Ok)."""
    m = len(commitments) // 32
    rc = host_lib().bph_rangeproof_verify(ctx._h, gens._h, gens.gens_capacity, gens.party_capacity, transcript.to_bytes(), proof, len(proof), commitments, m, n)
    if rc < 0:
        raise BpError(rc, lib().bp_last_error(ctx._h).decode())
    return rc


def ipp_create(ctx: Context, transcript: Transcript, Q: bytes, Gf: bytes, Hf: bytes, G: bytes, H: bytes, a: bytes, b: bytes):
    """InnerProductProof::create; returns the proof bytes (L_0,R_0,...,a,b) and advances the transcript."""
    n = len(a) // 32
    out = ctypes.create_string_buffer(32 * (2 * (n.bit_length() - 1) + 2))
    rc = host_lib().bph_ipp_create(ctx._h, transcript.state, Q, Gf, Hf, G, H, a, b, n, out)
    if rc != 0:
        raise BpError(rc, lib().bp_last_error(ctx._h).decode())
    return out.raw


def ipp_verify(ctx: Context, transcript: Transcript, n: int, Gf: bytes, Hf: bytes, P: bytes, Q: bytes, G: bytes, H: bytes, proof: bytes) -> int:
    rc = host_lib().bph_ipp_verify(ctx._h, transcript.state, n, Gf, Hf, P, Q, G, H, proof, len(proof))
    if rc < 0:
        raise BpError(rc, lib().bp_last_error(ctx._h).decode())
    return rc


def linear_create(ctx: Context, transcript: Transcript, seed: bytes, C: bytes, r: bytes, a: bytes, b: bytes, G: bytes, F: bytes, B: bytes):
    """LinearProof::create with rng = ChaChaRng::from_seed(seed); returns (status, proof bytes)."""
    n = len(a) // 32
    out = ctypes.create_string_buffer(32 * (2 * (n.bit_length() - 1) + 3))
    rc = host_lib().bph_linear_create(ctx._h, transcript.state, seed, C, r, a, b, G, F, B, n, out)
    if rc < 0:
        raise BpError(rc, lib().bp_last_error(ctx._h).decode())
    return rc, out.raw


def linear_verify(ctx: Context, transcript: Transcript, proof: bytes, C: bytes, G: bytes, F: bytes, B: bytes, b: bytes) -> int:
    rc = host_lib().bph_linear_verify(ctx._h, transcript.state, proof, len(proof), C, G, F, B, b, len(b) // 32)
    if rc < 0:
        raise BpError(rc, lib().bp_last_error(ctx._h).decode())
    return rc


def rangeproof_size(n: int, m: int) -> int:
    return 32 * (9 + 2 * ((n * m).bit_length() - 1))


def verify_batch(ctx: Context, gens: Gens, transcript: Transcript, proofs: bytes, commitments: bytes, n: int, m: int,
                 count: int, proof_len: int = None, seed: bytes = None):
    """RangeProof::verify_multiple for `count` proofs; returns the list of per-proof verdict codes."""
    if proof_len is None:
        proof_len = len(proofs) // count
    if len(proofs) != proof_len * count or len(commitments) != 32 * m * count:
        raise BpError(ERR_LENGTH_MISMATCH, "proof/commitment buffer sizes")
    verdicts = ctypes.create_string_buffer(count)
    ctx._check(lib().bp_rangeproof_verify_batch(ctx._h, gens._h, transcript.to_bytes(), proofs, proof_len, commitments, n, m, count, seed, verdicts))
    return list(verdicts.raw)


def verify_group(ctx: Context, gens: Gens, transcript: Transcript, proofs: bytes, commitments: bytes, n: int, m: int, count: int, n_batches: int, seed: bytes = None):
    """`n_batches` independent batches of `count` proofs in one launch group; returns (per-proof verdict codes, per-batch accept flags)."""
    proof_len = rangeproof_size(n, m)
    if len(proofs) != proof_len * count * n_batches or len(commitments) != 32 * m * count * n_batches:
        raise BpError(ERR_LENGTH_MISMATCH, "proof/commitment buffer sizes")
    verdicts = ctypes.create_string_buffer(count * n_batches); ok = ctypes.create_string_buffer(b"\xff" * n_batches, n_batches)      # every flag is written by _finish
    ctx._check(lib().bp_rangeproof_verify_group_begin(ctx._h, gens._h, transcript.to_bytes(), proofs, proof_len, commitments, n, m, count, n_batches, seed))
    ctx._check(lib().bp_rangeproof_verify_group_finish(ctx._h, verdicts, ok))
    return list(verdicts.raw), list(ok.raw)


# ---- aggregated range-proof MPC (bulletproofs_b200/host/mpc.{hpp,cpp}: Party / Dealer typestates of src/range_proof/{party,dealer,messages}.rs).
# Stateless harness form: a party is (v, v_blinding, n, j, ChaCha seed); wire layouts BitCommitment = V_j|A_j|S_j (96 B),
# PolyCommitment = T_1_j|T_2_j (64 B), ProofShare = t_x|t_x_blinding|e_blinding|l_vec|r_vec (32*(3+2n) B).  Status codes: MPC_* below.
MPC_OK, MPC_INVALID_BITSIZE, MPC_INVALID_GENERATORS_LENGTH, MPC_INVALID_AGGREGATION, MPC_MALICIOUS_DEALER, MPC_MALFORMED_PROOF_SHARES = 0, 3, 4, 5, 8, 10


def _mpc_rc(ctx, rc):
    if rc < 0:
        raise BpError(rc, lib().bp_last_error(ctx._h).decode())
    return rc


def mpc_party_bit_commitment(ctx, gens, v: int, v_blinding: bytes, n: int, j: int, seed: bytes):
    """Party::new + assign_position_with_rng(j, ChaChaRng::from_seed(seed)) -> (status, BitCommitment bytes)."""
    out = ctypes.create_string_buffer(96)
    rc = host_lib().bph_mpc_party_bit_commitment(ctx._h, gens._h, gens.gens_capacity, gens.party_capacity, v, v_blinding, n, j, seed, out)
    return _mpc_rc(ctx, rc), out.raw


def mpc_party_poly_commitment(ctx, gens, v: int, n: int, j: int, seed: bytes, y: bytes, z: bytes):
    """... + apply_challenge_with_rng(BitChallenge{y, z}) -> (status, PolyCommitment bytes)."""
    out = ctypes.create_string_buffer(64)
    rc = host_lib().bph_mpc_party_poly_commitment(ctx._h, gens._h, gens.gens_capacity, gens.party_capacity, v, n, j, seed, y, z, out)
    return _mpc_rc(ctx, rc), out.raw


def mpc_party_proof_share(ctx, gens, v: int, v_blinding: bytes, n: int, j: int, seed: bytes, y: bytes, z: bytes, x: bytes):
    """... + apply_challenge(PolyChallenge{x}) -> (status, ProofShare bytes); x = 0 -> MPC_MALICIOUS_DEALER."""
    out = ctypes.create_string_buffer(32 * (3 + 2 * n))
    rc = host_lib().bph_mpc_party_proof_share(ctx._h, gens._h, gens.gens_capacity, gens.party_capacity, v, v_blinding, n, j, seed, y, z, x, out)
    return _mpc_rc(ctx, rc), out.raw


def mpc_audit_share(ctx, gens, n: int, j: int, bit_commitment: bytes, y: bytes, z: bytes, poly_commitment: bytes, x: bytes, share: bytes) -> int:
    """ProofShare::audit_share (messages.rs:84-167): 0 = Ok, 1 = Err."""
    rc = host_lib().bph_mpc_audit_share(ctx._h, gens._h, gens.gens_capacity, gens.party_capacity, n, j, bit_commitment, y, z, poly_commitment, x, share)
    return _mpc_rc(ctx, rc)


def mpc_dealer_run(ctx, gens, transcript: Transcript, n: int, m: int, bit_commitments: bytes, poly_commitments: bytes = None, shares: bytes = None, trusted: bool = False):
    """Dealer::new -> receive_bit_commitments [-> receive_poly_commitments [-> receive_shares | receive_trusted_shares]] over the messages given.
    Returns (status, proof bytes or None, bad share flags, (y, z, x)); the transcript is advanced like the reference's &mut Transcript."""
    proof = ctypes.create_string_buffer(rangeproof_size(n, m)); bad = ctypes.create_string_buffer(max(m, 1)); ch = ctypes.create_string_buffer(96)
    rc = host_lib().bph_mpc_dealer_run(ctx._h, gens._h, gens.gens_capacity, gens.party_capacity, transcript.state, n, m, bit_commitments, poly_commitments, shares,
                                       int(trusted), proof, bad, ch)
    _mpc_rc(ctx, rc)
    done = rc == 0 and shares is not None
    return rc, (proof.raw if done else None), list(bad.raw[:m]), (ch.raw[:32], ch.raw[32:64], ch.raw[64:96])
