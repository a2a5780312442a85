"""ctypes binding of include/lwkzg.h (see package docstring)."""
from __future__ import annotations

import ctypes
import os
from typing import List, Optional, Sequence, Tuple

C_KZG_OK, C_KZG_BADARGS, C_KZG_ERROR, C_KZG_MALLOC = 0, 1, 2, 3
BYTES_PER_BLOB = 4096 * 32

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class KzgError(Exception):
    """A C ABI call returned something other than C_KZG_OK."""

    def __init__(self, code: int, where: str, detail: str = ""):
        super().__init__("%s -> C_KZG_RET %d%s" % (where, code, (": " + detail) if detail else ""))
        self.code = code


class _FFTSettings(ctypes.Structure):
    _fields_ = [("max_width", ctypes.c_uint64), ("expanded_roots_of_unity", ctypes.c_void_p),
                ("reverse_roots_of_unity", ctypes.c_void_p), ("roots_of_unity", ctypes.c_void_p)]


class CKZGSettings(ctypes.Structure):
    """KZGSettings, /root/reference/src/lib.rs:210-222."""
    _fields_ = [("fs", ctypes.c_void_p), ("g1_values", ctypes.c_void_p), ("g2_values", ctypes.c_void_p)]


def lib_path() -> str:
    return os.environ.get("LWKZG_LIB", os.path.join(_HERE, "liblwkzg_b200.so"))


def load_library() -> ctypes.CDLL:
    """Load liblwkzg_b200.so; raises if it has not been built (no fallback)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise RuntimeError("%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)" % path)
    lib = ctypes.CDLL(path)
    vp, sz, ip = ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_int)
    sp = ctypes.POINTER(CKZGSettings)
    bp = ctypes.POINTER(ctypes.c_bool)
    sig = {
        "load_trusted_setup": [sp, vp, sz, vp, sz],
        "load_trusted_setup_file": [sp, vp],
        "lwkzg_load_trusted_setup_ckzg": [sp, vp, ctypes.c_uint64, vp, ctypes.c_uint64, vp, ctypes.c_uint64, ctypes.c_uint64],
        "lwkzg_load_trusted_setup_file_ckzg": [sp, vp, ctypes.c_uint64],
        "lwkzg_last_load_times": [ctypes.POINTER(ctypes.c_double)] * 4,
        "free_trusted_setup": [sp],
        "blob_to_kzg_commitment": [vp, vp, sp],
        "compute_kzg_proof": [vp, vp, vp, vp, sp],
        "compute_blob_kzg_proof": [vp, vp, vp, sp],
        "verify_kzg_proof": [bp, vp, vp, vp, vp, sp],
        "verify_blob_kzg_proof": [bp, vp, vp, vp, sp],
        "verify_blob_kzg_proof_batch": [bp, vp, vp, vp, sz, sp],
        "lwkzg_blob_to_kzg_commitment_batch": [vp, vp, sz, sp, ip],
        "lwkzg_compute_blob_kzg_proof_batch": [vp, vp, vp, sz, sp, ip],
        "lwkzg_compute_kzg_proof_batch": [vp, vp, vp, vp, sz, sp, ip],
        "lwkzg_commit_and_prove_batch": [vp, vp, vp, sz, sp, ip],
        "lwkzg_commit_and_prove_batch_device": [vp, vp, vp, sz, sp, vp, vp],
        "lwkzg_blob_to_kzg_commitment_batch_device": [vp, vp, sz, sp, vp, vp],
        "lwkzg_verify_blob_kzg_proof_batch_device": [bp, vp, vp, vp, sz, sp],
        "lwkzg_verify_kzg_proofs": [bp, vp, vp, vp, vp, sz, sp, ip],
        "lwkzg_verify_kzg_proofs_device": [vp, vp, vp, vp, vp, sz, sp, vp, vp],
        "lwkzg_verify_blob_kzg_proof_batches": [bp, vp, vp, vp, vp, sz, sp, ip],
        "lwkzg_verify_blob_kzg_proof_batches_device": [vp, vp, vp, vp, vp, sz, sp, vp, vp],
        "lwkzg_debug_blob_batch_challenges": [vp, sz, sp],
        "lwkzg_compute_blob_kzg_proof_batch_device": [vp, vp, vp, sz, sp, vp, vp],
        "lwkzg_g1_lincomb": [vp, vp, vp, sz],
        "lwkzg_verify_batch_phase1": [vp, vp, vp, vp, sz, sp],
        "lwkzg_verify_batch_phase2": [vp, vp, sz, sz, sz, sp],
        "lwkzg_verify_batch_phase3": [bp, vp, sz, sp],
        "lwkzg_verify_batch_phase1_device": [vp, vp, vp, vp, sz, ctypes.c_int, sp],
        "lwkzg_verify_batch_phase2_device": [vp, vp, sz, sz, sz, sp],
        "lwkzg_verify_batch_phase3_device": [bp, vp, sz, sp],
        "lwkzg_set_devices": [ip, ctypes.c_int],
        "lwkzg_get_devices": [ip, ctypes.c_int],
        "lwkzg_debug_batch_challenge": [vp, sp],
        "lwkzg_synth_blobs_device": [vp, ctypes.c_uint64, sz, vp],
        "lwkzg_synth_blob_host": [vp, ctypes.c_uint64],
        "compute_cells_and_kzg_proofs": [vp, vp, vp, sp],
        "recover_cells_and_kzg_proofs": [vp, vp, vp, vp, sz, sp],
        "verify_cell_kzg_proof_batch": [bp, vp, vp, vp, vp, sz, sp],
        "lwkzg_compute_cells_and_kzg_proofs_batch": [vp, vp, vp, sz, sp, ip],
        "lwkzg_compute_cells_and_kzg_proofs_batch_device": [vp, vp, vp, sz, sp, vp, vp],
        "lwkzg_commit_and_compute_cells_and_kzg_proofs_batch": [vp, vp, vp, vp, sz, sp, ip],
        "lwkzg_commit_and_compute_cells_and_kzg_proofs_batch_device": [vp, vp, vp, vp, sz, sp, vp, vp],
        "lwkzg_recover_cells_and_kzg_proofs_batch": [vp, vp, vp, vp, sz, sz, sp, ip],
        "lwkzg_recover_cells_and_kzg_proofs_batch_device": [vp, vp, vp, vp, sz, sz, sp, vp, vp],
        "lwkzg_verify_cell_kzg_proof_batches": [bp, vp, vp, vp, vp, vp, sz, sp, ip],
        "lwkzg_verify_cell_kzg_proof_batches_device": [vp, vp, vp, vp, vp, vp, sz, sp, vp, vp],
        "lwkzg_verify_blob_cell_kzg_proof_batches": [bp, vp, vp, vp, vp, sz, sp, ip],
        "lwkzg_verify_blob_cell_kzg_proof_batches_device": [vp, vp, vp, vp, vp, sz, sp, vp, vp],
        "lwkzg_debug_cell_batch_challenges": [vp, sz, sp],
        "lwkzg_cell_window_bits": [sp],
        "lwkzg_table_share": [sp],
        "lwkzg_debug_cell_stages": [vp, vp, vp, vp, vp, sp],
        "lwkzg_set_option": [ctypes.c_char_p, ctypes.c_long],
        "lwkzg_get_option": [ctypes.c_char_p],
    }
    for name, args in sig.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = ctypes.c_int
    lib.lwkzg_synth_blob_host.restype = None
    lib.lwkzg_get_option.restype = ctypes.c_long
    lib.lwkzg_imad_peak.argtypes = [ctypes.c_int]
    lib.lwkzg_imad_peak.restype = ctypes.c_double
    lib.lwkzg_bench_msm_kernel.argtypes = [vp, sz, ctypes.c_int, ctypes.c_int, sp]
    lib.lwkzg_bench_msm_kernel.restype = ctypes.c_double
    lib.lwkzg_bench_var_msm.argtypes = [vp, sz, ctypes.c_int, ctypes.c_uint64, sp]
    lib.lwkzg_bench_var_msm.restype = ctypes.c_double
    lib.lwkzg_bench_pairing.argtypes = [ctypes.c_int, sp]
    lib.lwkzg_bench_pairing.restype = ctypes.c_double
    lib.lwkzg_window_bits.argtypes = [sp]
    lib.lwkzg_window_bits.restype = ctypes.c_int
    lib.lwkzg_kernel_launches.argtypes = []
    lib.lwkzg_kernel_launches.restype = ctypes.c_uint64
    lib.lwkzg_last_error.argtypes = []
    lib.lwkzg_last_error.restype = ctypes.c_char_p
    lib.lwkzg_version.argtypes = []
    lib.lwkzg_version.restype = ctypes.c_char_p
    _LIB = lib
    return lib


def last_error() -> str:
    return load_library().lwkzg_last_error().decode()


def _check(code: int, where: str):
    if code != C_KZG_OK:
        raise KzgError(code, where, last_error())


def set_option(name: str, value: int):
    if load_library().lwkzg_set_option(name.encode(), int(value)) != 0:
        raise ValueError("bad option %s=%r" % (name, value))


def get_option(name: str) -> int:
    return int(load_library().lwkzg_get_option(name.encode()))


def kernel_launches() -> int:
    return int(load_library().lwkzg_kernel_launches())


def imad_peak(variant: int = 0) -> float:
    """Measured MAC32/s of the integer pipe (roofline denominator R_int)."""
    return float(load_library().lwkzg_imad_peak(variant))


class Settings:
    """Owns a C ``KZGSettings`` produced by the library's loaders."""

    def __init__(self):
        self.c = CKZGSettings()
        self._loaded = False

    @property
    def ptr(self):
        return ctypes.byref(self.c)

    def free(self):
        if self._loaded:
            load_library().free_trusted_setup(self.ptr)
            self._loaded = False

    def g1_values_bytes(self) -> bytes:
        return ctypes.string_at(self.c.g1_values, 4096 * 144)

    def g2_values_bytes(self) -> bytes:
        return ctypes.string_at(self.c.g2_values, 65 * 288)

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _load_from_file(path: str, fn: str, *extra) -> Settings:
    lib = load_library()
    libc = ctypes.CDLL(None)
    libc.fopen.restype = ctypes.c_void_p
    libc.fopen.argtypes = [ctypes.c_char_p, ctypes.c_char_p]
    libc.fclose.argtypes = [ctypes.c_void_p]
    fp = libc.fopen(path.encode(), b"rb")
    if not fp:
        raise FileNotFoundError(path)
    s = Settings()
    try:
        _check(getattr(lib, fn)(s.ptr, fp, *extra), fn)
    finally:
        libc.fclose(fp)
    s._loaded = True
    return s


def load_trusted_setup_file(path: str) -> Settings:
    """load_trusted_setup_file(KZGSettings*, FILE*) -- lib.rs:779-802.  Reads the reference's format (monomial G1
    points first); a c-kzg-4844 trusted_setup.txt needs load_trusted_setup_file_ckzg."""
    return _load_from_file(path, "load_trusted_setup_file")


def load_trusted_setup_file_ckzg(path: str, precompute: int = 0) -> Settings:
    """c-kzg-4844's trusted_setup.txt (4096 Lagrange G1, 65 G2, 4096 monomial G1 points), checked on the device to be
    one powers-of-tau setup -- lwkzg_load_trusted_setup_file_ckzg."""
    return _load_from_file(path, "lwkzg_load_trusted_setup_file_ckzg", precompute)


def load_trusted_setup_ckzg(g1_monomial: bytes, g1_lagrange: bytes, g2_monomial: bytes, precompute: int = 0) -> Settings:
    """c-kzg-4844 v2's load_trusted_setup(out, g1_monomial, ..., g1_lagrange, ..., g2_monomial, ..., precompute): the
    three compressed sections as bytes -- lwkzg_load_trusted_setup_ckzg."""
    lib = load_library()
    s = Settings()
    _check(lib.lwkzg_load_trusted_setup_ckzg(s.ptr, g1_monomial, len(g1_monomial), g1_lagrange, len(g1_lagrange), g2_monomial, len(g2_monomial),
                                             precompute), "lwkzg_load_trusted_setup_ckzg")
    s._loaded = True
    return s


def last_load_times() -> dict:
    """Phase times (ms) of this thread's last trusted-setup load: decode, check, convert, build."""
    v = [ctypes.c_double() for _ in range(4)]
    load_library().lwkzg_last_load_times(*[ctypes.byref(x) for x in v])
    return dict(zip(("decode_ms", "check_ms", "convert_ms", "build_ms"), (x.value for x in v)))


def load_trusted_setup(g1_bytes: bytes, g2_bytes: bytes, n1: Optional[int] = None, n2: Optional[int] = None) -> Settings:
    """load_trusted_setup -- lib.rs:709-776."""
    lib = load_library()
    n1 = len(g1_bytes) // 48 if n1 is None else n1
    n2 = len(g2_bytes) // 96 if n2 is None else n2
    s = Settings()
    _check(lib.load_trusted_setup(s.ptr, g1_bytes, n1, g2_bytes, n2), "load_trusted_setup")
    s._loaded = True
    return s


def _sp(s):
    return s.ptr if isinstance(s, Settings) else ctypes.byref(s)


def blob_to_kzg_commitment(blob: bytes, s) -> bytes:
    assert len(blob) == BYTES_PER_BLOB
    out = ctypes.create_string_buffer(48)
    _check(load_library().blob_to_kzg_commitment(out, blob, _sp(s)), "blob_to_kzg_commitment")
    return out.raw


def compute_kzg_proof(blob: bytes, z_bytes: bytes, s) -> Tuple[bytes, bytes]:
    assert len(blob) == BYTES_PER_BLOB and len(z_bytes) == 32
    proof = ctypes.create_string_buffer(48)
    y = ctypes.create_string_buffer(32)
    _check(load_library().compute_kzg_proof(proof, y, blob, z_bytes, _sp(s)), "compute_kzg_proof")
    return proof.raw, y.raw


def compute_blob_kzg_proof(blob: bytes, commitment: bytes, s) -> bytes:
    assert len(blob) == BYTES_PER_BLOB and len(commitment) == 48
    out = ctypes.create_string_buffer(48)
    _check(load_library().compute_blob_kzg_proof(out, blob, commitment, _sp(s)), "compute_blob_kzg_proof")
    return out.raw


def verify_kzg_proof(commitment: bytes, z_bytes: bytes, y_bytes: bytes, proof: bytes, s) -> bool:
    ok = ctypes.c_bool(False)
    _check(load_library().verify_kzg_proof(ctypes.byref(ok), commitment, z_bytes, y_bytes, proof, _sp(s)), "verify_kzg_proof")
    return bool(ok.value)


def verify_kzg_proofs(commitments: Sequence[bytes], zs: Sequence[bytes], ys: Sequence[bytes], proofs: Sequence[bytes], s) -> Tuple[List[bool], List[int]]:
    """n independent verify_kzg_proof checks in one call -> (verdict list, status list): for each item the verdict and
    code verify_kzg_proof returns for it (a failed item has verdict False)."""
    n = len(commitments)
    assert len(zs) == len(ys) == len(proofs) == n
    oks = (ctypes.c_bool * max(1, n))()
    st = _status_list(n)
    _check(load_library().lwkzg_verify_kzg_proofs(oks, _cat(commitments, 48) or b"\0", _cat(zs, 32) or b"\0", _cat(ys, 32) or b"\0",
                                                  _cat(proofs, 48) or b"\0", n, _sp(s), st), "lwkzg_verify_kzg_proofs")
    return [bool(oks[i]) for i in range(n)], list(st)[:n]


def verify_kzg_proofs_device(d_ok: int, d_commitments: int, d_zs: int, d_ys: int, d_proofs: int, n: int, s, stream: int = 0, d_status: int = 0):
    """All buffers are raw device addresses (torch: tensor.data_ptr()); d_ok and d_status (0 = not wanted) are n int32
    each.  Asynchronous on `stream`."""
    _check(load_library().lwkzg_verify_kzg_proofs_device(d_ok or None, d_commitments or None, d_zs or None, d_ys or None, d_proofs or None, n, _sp(s),
                                                         stream or None, d_status or None), "lwkzg_verify_kzg_proofs_device")


def verify_blob_kzg_proof(blob: bytes, commitment: bytes, proof: bytes, s) -> bool:
    ok = ctypes.c_bool(False)
    _check(load_library().verify_blob_kzg_proof(ctypes.byref(ok), blob, commitment, proof, _sp(s)), "verify_blob_kzg_proof")
    return bool(ok.value)


def _cat(items: Sequence[bytes], each: int) -> bytes:
    b = b"".join(items)
    assert len(b) == each * len(items)
    return b


def verify_blob_kzg_proof_batch(blobs: Sequence[bytes], commitments: Sequence[bytes], proofs: Sequence[bytes], s) -> bool:
    n = len(blobs)
    ok = ctypes.c_bool(False)
    code = load_library().verify_blob_kzg_proof_batch(ctypes.byref(ok), _cat(blobs, BYTES_PER_BLOB), _cat(commitments, 48), _cat(proofs, 48), n, _sp(s))
    _check(code, "verify_blob_kzg_proof_batch")
    return bool(ok.value)


def verify_blob_kzg_proof_batch_ptr(blobs_ptr: int, commitments_ptr: int, proofs_ptr: int, n: int, s) -> bool:
    """Same C call with raw host addresses (e.g. pinned torch tensors): no Python-side copies."""
    ok = ctypes.c_bool(False)
    _check(load_library().verify_blob_kzg_proof_batch(ctypes.byref(ok), blobs_ptr, commitments_ptr, proofs_ptr, n, _sp(s)), "verify_blob_kzg_proof_batch")
    return bool(ok.value)


def verify_blob_kzg_proof_batch_device(d_blobs: int, d_commitments: int, d_proofs: int, n: int, s) -> bool:
    """verify_blob_kzg_proof_batch with the inputs already in device memory (raw device addresses)."""
    ok = ctypes.c_bool(False)
    _check(load_library().lwkzg_verify_blob_kzg_proof_batch_device(ctypes.byref(ok), d_blobs, d_commitments, d_proofs, n, _sp(s)),
           "lwkzg_verify_blob_kzg_proof_batch_device")
    return bool(ok.value)


def _offsets(offsets: Sequence[int]):
    """The K + 1 batch offsets of a per-batch call as the uint64 array the C calls take."""
    return (ctypes.c_uint64 * max(1, len(offsets)))(*offsets)


def _debug_challenges(fn: str, n_batches: int, s) -> List[int]:
    """The 32-byte little-endian challenges of the last call of a per-batch family, read by the C test hook `fn`."""
    out = ctypes.create_string_buffer(32 * max(1, n_batches))
    _check(getattr(load_library(), fn)(out, n_batches, _sp(s)), fn)
    return [int.from_bytes(out.raw[32 * i: 32 * i + 32], "little") for i in range(n_batches)]


def verify_blob_kzg_proof_batches(batches: Sequence[Tuple[Sequence[bytes], Sequence[bytes], Sequence[bytes]]], s) -> Tuple[List[bool], List[int]]:
    """K independent verify_blob_kzg_proof_batch checks in one call.  batches: (blobs, commitments, proofs) per batch ->
    (verdict list, status list): per batch, what verify_blob_kzg_proof_batch over that batch alone returns."""
    k = len(batches)
    offsets = [0]
    for bl, com, pr in batches:
        assert len(bl) == len(com) == len(pr)
        offsets.append(offsets[-1] + len(bl))
    off = _offsets(offsets)
    oks = (ctypes.c_bool * max(1, k))()
    st = _status_list(k)
    _check(load_library().lwkzg_verify_blob_kzg_proof_batches(oks, b"".join(_cat(b[0], BYTES_PER_BLOB) for b in batches) or b"\0",
                                                              b"".join(_cat(b[1], 48) for b in batches) or b"\0",
                                                              b"".join(_cat(b[2], 48) for b in batches) or b"\0", off, k, _sp(s), st),
           "lwkzg_verify_blob_kzg_proof_batches")
    return [bool(oks[i]) for i in range(k)], list(st)[:k]


def verify_blob_kzg_proof_batches_device(d_ok: int, d_blobs: int, d_commitments: int, d_proofs: int, offsets: Sequence[int], s, stream: int = 0,
                                         d_status: int = 0):
    """All buffers are raw device addresses (torch: tensor.data_ptr()) except offsets (K + 1 host integers, in blobs);
    d_ok and d_status (0 = not wanted) are K int32 each.  Asynchronous on `stream`."""
    k = len(offsets) - 1
    off = _offsets(offsets)
    _check(load_library().lwkzg_verify_blob_kzg_proof_batches_device(d_ok or None, d_blobs or None, d_commitments or None, d_proofs or None, off, k,
                                                                     _sp(s), stream or None, d_status or None),
           "lwkzg_verify_blob_kzg_proof_batches_device")


def debug_blob_batch_challenges(n_batches: int, s) -> List[int]:
    """The challenges r_b the last verify_blob_kzg_proof_batches[_device] call derived (0 for batches of fewer than two
    blobs; test hook)."""
    return _debug_challenges("lwkzg_debug_blob_batch_challenges", n_batches, s)


# ------------------------------------------------------------------ batch extensions (host buffers)
def _status_list(n):
    return (ctypes.c_int * max(n, 1))()


def blob_to_kzg_commitment_batch(blobs: bytes, n: int, s) -> Tuple[List[bytes], List[int]]:
    out = ctypes.create_string_buffer(48 * max(n, 1))
    st = _status_list(n)
    _check(load_library().lwkzg_blob_to_kzg_commitment_batch(out, blobs, n, _sp(s), st), "lwkzg_blob_to_kzg_commitment_batch")
    return [out.raw[48 * i: 48 * i + 48] for i in range(n)], list(st)[:n]


def compute_blob_kzg_proof_batch(blobs: bytes, commitments: bytes, n: int, s) -> Tuple[List[bytes], List[int]]:
    out = ctypes.create_string_buffer(48 * max(n, 1))
    st = _status_list(n)
    _check(load_library().lwkzg_compute_blob_kzg_proof_batch(out, blobs, commitments, n, _sp(s), st), "lwkzg_compute_blob_kzg_proof_batch")
    return [out.raw[48 * i: 48 * i + 48] for i in range(n)], list(st)[:n]


def compute_kzg_proof_batch(blobs: bytes, zs: bytes, n: int, s):
    proofs = ctypes.create_string_buffer(48 * max(n, 1))
    ys = ctypes.create_string_buffer(32 * max(n, 1))
    st = _status_list(n)
    _check(load_library().lwkzg_compute_kzg_proof_batch(proofs, ys, blobs, zs, n, _sp(s), st), "lwkzg_compute_kzg_proof_batch")
    return ([proofs.raw[48 * i: 48 * i + 48] for i in range(n)], [ys.raw[32 * i: 32 * i + 32] for i in range(n)], list(st)[:n])


def commit_and_prove_batch(blobs, n: int, s, out_commitments=None, out_proofs=None):
    """blobs / outputs may be bytes-like objects or integer host addresses
    (e.g. a pinned torch tensor's data_ptr())."""
    lib = load_library()
    own = out_commitments is None
    if own:
        out_commitments = ctypes.create_string_buffer(48 * max(n, 1))
        out_proofs = ctypes.create_string_buffer(48 * max(n, 1))
    st = _status_list(n)
    _check(lib.lwkzg_commit_and_prove_batch(out_commitments, out_proofs, blobs, n, _sp(s), st), "lwkzg_commit_and_prove_batch")
    if own:
        return ([out_commitments.raw[48 * i: 48 * i + 48] for i in range(n)],
                [out_proofs.raw[48 * i: 48 * i + 48] for i in range(n)], list(st)[:n])
    return list(st)[:n]


def g1_lincomb(points_xy_be: bytes, scalars_be: bytes, n: int) -> bytes:
    out = ctypes.create_string_buffer(48)
    _check(load_library().lwkzg_g1_lincomb(out, points_xy_be, scalars_be, n), "lwkzg_g1_lincomb")
    return out.raw


# ------------------------------------------------------------------ device-pointer helpers
def commit_and_prove_batch_device(d_commitments: int, d_proofs: int, d_blobs: int, n: int, s, stream: int = 0, d_status: int = 0):
    """All arguments are raw device addresses (torch: tensor.data_ptr()) and a
    cudaStream_t handle (torch: torch.cuda.current_stream().cuda_stream)."""
    _check(load_library().lwkzg_commit_and_prove_batch_device(d_commitments, d_proofs, d_blobs, n, _sp(s), stream, d_status),
           "lwkzg_commit_and_prove_batch_device")


def blob_to_kzg_commitment_batch_device(d_commitments: int, d_blobs: int, n: int, s, stream: int = 0, d_status: int = 0):
    _check(load_library().lwkzg_blob_to_kzg_commitment_batch_device(d_commitments, d_blobs, n, _sp(s), stream, d_status),
           "lwkzg_blob_to_kzg_commitment_batch_device")


def compute_blob_kzg_proof_batch_device(d_proofs: int, d_blobs: int, d_commitments: int, n: int, s, stream: int = 0, d_status: int = 0):
    _check(load_library().lwkzg_compute_blob_kzg_proof_batch_device(d_proofs, d_blobs, d_commitments, n, _sp(s), stream, d_status),
           "lwkzg_compute_blob_kzg_proof_batch_device")


def bench_msm_kernel(d_blobs: int, n: int, s, blocks_per_blob: int = 0, iters: int = 5) -> float:
    """Average ms per launch of the dominant kernel alone (roofline leg)."""
    ms = float(load_library().lwkzg_bench_msm_kernel(d_blobs, n, blocks_per_blob, iters, _sp(s)))
    if ms < 0:
        raise KzgError(C_KZG_ERROR, "lwkzg_bench_msm_kernel", last_error())
    return ms


def bench_var_msm(n: int, s, iters: int = 3, seed: int = 0):
    """(ms per MSM, compressed result) for the synthetic variable-base MSM of size n."""
    out = ctypes.create_string_buffer(48)
    ms = float(load_library().lwkzg_bench_var_msm(out, n, iters, seed, _sp(s)))
    if ms < 0:
        raise KzgError(C_KZG_ERROR, "lwkzg_bench_var_msm", last_error())
    return ms, out.raw


def bench_pairing(s, iters: int = 5) -> float:
    """ms per run of the partial-sum fold + 2-pairing check of the last batched verification on these settings."""
    ms = float(load_library().lwkzg_bench_pairing(iters, _sp(s)))
    if ms < 0:
        raise KzgError(C_KZG_ERROR, "lwkzg_bench_pairing", last_error())
    return ms


def window_bits(s) -> int:
    return int(load_library().lwkzg_window_bits(_sp(s)))


_X2 = 0xD201000000010000 ** 2          # BLS12-381: x^2, the GLV split modulus (csrc/recode.cuh)
_R = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001


def table_geometry(c: int):
    """(windows, [multiples stored per point for each window]) of the fixed-base digit table for window c --
    host mirror of csrc/recode.cuh."""
    w = -(-128 // c)
    counts = [1 << (c - 1)] * (w - 1) + [((_X2 - 1) >> (c * (w - 1))) + 1]
    return w, counts


def synth_point_dlogs(s, n: int, tau: int) -> List[int]:
    """Discrete logs (base G, mod r) of the n synthetic points bench_var_msm uses: point t is entry
    (t * 2654435761) mod entries of the fixed-base table, i.e. d * 2^(c j) * tau^i * G for a monomial setup
    (csrc/varmsm.cu vm_synth_kernel, csrc/table.cu layout)."""
    c = window_bits(s)
    w, counts = table_geometry(c)
    per_window = 4096 << (c - 1)
    entries = per_window * (w - 1) + 4096 * counts[-1]
    tau_pow = [1] * 4096
    for i in range(1, 4096):
        tau_pow[i] = tau_pow[i - 1] * tau % _R
    two_pow = [pow(2, c * j, _R) for j in range(w)]
    out = []
    for t in range(n):
        e = (t * 2654435761) % entries
        j = min(e // per_window, w - 1)
        off = e - j * per_window
        i, d = divmod(off, counts[j])
        out.append((d + 1) * two_pow[j] * tau_pow[i] % _R)
    return out


def synth_blobs_device(d_blobs: int, first_blob: int, n: int, stream: int = 0):
    _check(load_library().lwkzg_synth_blobs_device(d_blobs, first_blob, n, stream), "lwkzg_synth_blobs_device")


def synth_blob_host(k: int) -> bytes:
    buf = ctypes.create_string_buffer(BYTES_PER_BLOB)
    load_library().lwkzg_synth_blob_host(buf, k)
    return buf.raw


# ------------------------------------------------------------------ multi-GPU verification phases
def debug_batch_challenge(s) -> int:
    """The batch challenge r left by the last batched verification / phase 2 on these settings (test hook)."""
    out = ctypes.create_string_buffer(32)
    _check(load_library().lwkzg_debug_batch_challenge(out, _sp(s)), "lwkzg_debug_batch_challenge")
    return int.from_bytes(out.raw, "little")


def verify_batch_phase1(blobs: bytes, commitments: bytes, proofs: bytes, n_local: int, s) -> bytes:
    out = ctypes.create_string_buffer(160 * max(n_local, 1))
    _check(load_library().lwkzg_verify_batch_phase1(out, blobs, commitments, proofs, n_local, _sp(s)), "lwkzg_verify_batch_phase1")
    return out.raw[: 160 * n_local]


def verify_batch_phase2(all_tuples: bytes, n_total: int, first: int, n_local: int, s) -> bytes:
    out = ctypes.create_string_buffer(288)
    _check(load_library().lwkzg_verify_batch_phase2(out, all_tuples, n_total, first, n_local, _sp(s)), "lwkzg_verify_batch_phase2")
    return out.raw


def verify_batch_phase1_device(d_tuples: int, blobs_ptr: int, commitments_ptr: int, proofs_ptr: int, n_local: int, s, inputs_on_device: bool):
    """phase 1 with the tuples written to device memory (d_tuples: n_local x 160 bytes); inputs are raw host or device addresses."""
    _check(load_library().lwkzg_verify_batch_phase1_device(d_tuples, blobs_ptr, commitments_ptr, proofs_ptr, n_local, 1 if inputs_on_device else 0, _sp(s)),
           "lwkzg_verify_batch_phase1_device")


def verify_batch_phase2_device(d_partial: int, d_all_tuples: int, n_total: int, first: int, n_local: int, s):
    _check(load_library().lwkzg_verify_batch_phase2_device(d_partial, d_all_tuples, n_total, first, n_local, _sp(s)), "lwkzg_verify_batch_phase2_device")


def verify_batch_phase3_device(d_partials: int, n_ranks: int, s) -> bool:
    ok = ctypes.c_bool(False)
    _check(load_library().lwkzg_verify_batch_phase3_device(ctypes.byref(ok), d_partials, n_ranks, _sp(s)), "lwkzg_verify_batch_phase3_device")
    return bool(ok.value)


def set_devices(ids: Sequence[int]):
    """lwkzg_set_devices: shard the host-buffer batch calls of THIS process over the listed GPUs ([] = default)."""
    arr = (ctypes.c_int * max(len(ids), 1))(*ids)
    if load_library().lwkzg_set_devices(arr, len(ids)) != 0:
        raise ValueError("lwkzg_set_devices(%r) rejected" % (list(ids),))


def get_devices() -> List[int]:
    arr = (ctypes.c_int * 64)()
    n = load_library().lwkzg_get_devices(arr, 64)
    return [arr[i] for i in range(min(n, 64))]


def verify_batch_phase3(partials: bytes, n_ranks: int, s) -> bool:
    ok = ctypes.c_bool(False)
    _check(load_library().lwkzg_verify_batch_phase3(ctypes.byref(ok), partials, n_ranks, _sp(s)), "lwkzg_verify_batch_phase3")
    return bool(ok.value)


# ------------------------------------------------------------------ PeerDAS / EIP-7594 cells (include/lwkzg.h part 3)
CELLS_PER_EXT_BLOB = 128
BYTES_PER_CELL = 2048


def compute_cells_and_kzg_proofs(blob: bytes, s, want_cells: bool = True, want_proofs: bool = True) -> Tuple[List[bytes], List[bytes]]:
    """compute_cells_and_kzg_proofs of c-kzg-4844's eip7594 API: 128 cells and / or 128 proofs of one blob."""
    assert len(blob) == BYTES_PER_BLOB
    cells = ctypes.create_string_buffer(CELLS_PER_EXT_BLOB * BYTES_PER_CELL) if want_cells else None
    proofs = ctypes.create_string_buffer(CELLS_PER_EXT_BLOB * 48) if want_proofs else None
    _check(load_library().compute_cells_and_kzg_proofs(cells, proofs, blob, _sp(s)), "compute_cells_and_kzg_proofs")
    cl = [cells.raw[i * BYTES_PER_CELL: (i + 1) * BYTES_PER_CELL] for i in range(CELLS_PER_EXT_BLOB)] if want_cells else []
    pl = [proofs.raw[i * 48: (i + 1) * 48] for i in range(CELLS_PER_EXT_BLOB)] if want_proofs else []
    return cl, pl


def compute_cells_and_kzg_proofs_batch(blobs: bytes, n: int, s, want_cells: bool = True, want_proofs: bool = True):
    """-> (cells bytes n x 128 x 2048 or b"", proofs bytes n x 128 x 48 or b"", status list)."""
    assert len(blobs) == n * BYTES_PER_BLOB
    cells = ctypes.create_string_buffer(max(1, n * CELLS_PER_EXT_BLOB * BYTES_PER_CELL)) if want_cells else None
    proofs = ctypes.create_string_buffer(max(1, n * CELLS_PER_EXT_BLOB * 48)) if want_proofs else None
    st = (ctypes.c_int * max(1, n))()
    _check(load_library().lwkzg_compute_cells_and_kzg_proofs_batch(cells, proofs, blobs, n, _sp(s), st), "lwkzg_compute_cells_and_kzg_proofs_batch")
    return (cells.raw[: n * CELLS_PER_EXT_BLOB * BYTES_PER_CELL] if want_cells else b"", proofs.raw[: n * CELLS_PER_EXT_BLOB * 48] if want_proofs else b"",
            list(st)[:n])


def compute_cells_and_kzg_proofs_batch_device(d_cells: int, d_proofs: int, d_blobs: int, n: int, s, stream: int = 0, d_status: int = 0):
    """Device-pointer variant: raw device addresses (0 = not wanted), asynchronous with respect to the host."""
    _check(load_library().lwkzg_compute_cells_and_kzg_proofs_batch_device(d_cells or None, d_proofs or None, d_blobs, n, _sp(s), stream or None,
                                                                          d_status or None), "lwkzg_compute_cells_and_kzg_proofs_batch_device")


def commit_and_compute_cells_and_kzg_proofs_batch(blobs: bytes, n: int, s, want_cells: bool = False):
    """-> (commitments list, cells bytes n x 128 x 2048 or b"", proofs bytes n x 128 x 48, status list): each blob read
    once for its commitment, its 128 cell proofs and (want_cells) its cells."""
    assert len(blobs) == n * BYTES_PER_BLOB
    coms = ctypes.create_string_buffer(max(1, n * 48))
    cells = ctypes.create_string_buffer(max(1, n * CELLS_PER_EXT_BLOB * BYTES_PER_CELL)) if want_cells else None
    proofs = ctypes.create_string_buffer(max(1, n * CELLS_PER_EXT_BLOB * 48))
    st = (ctypes.c_int * max(1, n))()
    _check(load_library().lwkzg_commit_and_compute_cells_and_kzg_proofs_batch(coms, cells, proofs, blobs, n, _sp(s), st),
           "lwkzg_commit_and_compute_cells_and_kzg_proofs_batch")
    return ([coms.raw[48 * i: 48 * i + 48] for i in range(n)], cells.raw[: n * CELLS_PER_EXT_BLOB * BYTES_PER_CELL] if want_cells else b"",
            proofs.raw[: n * CELLS_PER_EXT_BLOB * 48], list(st)[:n])


def commit_and_compute_cells_and_kzg_proofs_batch_device(d_commitments: int, d_cells: int, d_proofs: int, d_blobs: int, n: int, s, stream: int = 0,
                                                         d_status: int = 0):
    """Device-pointer variant: raw device addresses (d_cells, d_status: 0 = not wanted), asynchronous with respect to
    the host."""
    _check(load_library().lwkzg_commit_and_compute_cells_and_kzg_proofs_batch_device(d_commitments or None, d_cells or None, d_proofs or None, d_blobs or None,
                                                                                     n, _sp(s), stream or None, d_status or None),
           "lwkzg_commit_and_compute_cells_and_kzg_proofs_batch_device")


def recover_cells_and_kzg_proofs(cell_indices: Sequence[int], cells: Sequence[bytes], s, want_cells: bool = True, want_proofs: bool = True):
    n = len(cell_indices)
    idx = (ctypes.c_uint64 * max(1, n))(*cell_indices)
    rc = ctypes.create_string_buffer(CELLS_PER_EXT_BLOB * BYTES_PER_CELL) if want_cells else None
    rp = ctypes.create_string_buffer(CELLS_PER_EXT_BLOB * 48) if want_proofs else None
    _check(load_library().recover_cells_and_kzg_proofs(rc, rp, idx, _cat(cells, BYTES_PER_CELL), n, _sp(s)), "recover_cells_and_kzg_proofs")
    cl = [rc.raw[i * BYTES_PER_CELL: (i + 1) * BYTES_PER_CELL] for i in range(CELLS_PER_EXT_BLOB)] if want_cells else []
    pl = [rp.raw[i * 48: (i + 1) * 48] for i in range(CELLS_PER_EXT_BLOB)] if want_proofs else []
    return cl, pl


def recover_cells_and_kzg_proofs_batch(cell_indices: Sequence[int], cells: bytes, num_cells: int, n: int, s, want_cells: bool = True,
                                       want_proofs: bool = True):
    """n blobs from num_cells cells each (indices and cells n x num_cells, blob-major)
    -> (cells bytes n x 128 x 2048 or b"", proofs bytes n x 128 x 48 or b"", status list)."""
    assert len(cell_indices) == n * num_cells and len(cells) == n * num_cells * BYTES_PER_CELL
    idx = (ctypes.c_uint64 * max(1, n * num_cells))(*cell_indices)
    rc = ctypes.create_string_buffer(max(1, n * CELLS_PER_EXT_BLOB * BYTES_PER_CELL)) if want_cells else None
    rp = ctypes.create_string_buffer(max(1, n * CELLS_PER_EXT_BLOB * 48)) if want_proofs else None
    st = (ctypes.c_int * max(1, n))()
    _check(load_library().lwkzg_recover_cells_and_kzg_proofs_batch(rc, rp, idx, cells or b"\0", num_cells, n, _sp(s), st),
           "lwkzg_recover_cells_and_kzg_proofs_batch")
    return (rc.raw[: n * CELLS_PER_EXT_BLOB * BYTES_PER_CELL] if want_cells else b"", rp.raw[: n * CELLS_PER_EXT_BLOB * 48] if want_proofs else b"",
            list(st)[:n])


def recover_cells_and_kzg_proofs_batch_device(d_cells_out: int, d_proofs_out: int, d_cell_indices: int, d_cells: int, num_cells: int, n: int, s,
                                              stream: int = 0, d_status: int = 0):
    """Device-pointer variant: raw device addresses (0 = not wanted), asynchronous with respect to the host."""
    _check(load_library().lwkzg_recover_cells_and_kzg_proofs_batch_device(d_cells_out or None, d_proofs_out or None, d_cell_indices or None,
                                                                          d_cells or None, num_cells, n, _sp(s), stream or None, d_status or None),
           "lwkzg_recover_cells_and_kzg_proofs_batch_device")


def verify_cell_kzg_proof_batch(commitments: Sequence[bytes], cell_indices: Sequence[int], cells: Sequence[bytes], proofs: Sequence[bytes], s) -> bool:
    n = len(cell_indices)
    assert len(commitments) == len(cells) == len(proofs) == n
    idx = (ctypes.c_uint64 * max(1, n))(*cell_indices)
    ok = ctypes.c_bool(False)
    _check(load_library().verify_cell_kzg_proof_batch(ctypes.byref(ok), _cat(commitments, 48) or b"\0", idx, _cat(cells, BYTES_PER_CELL) or b"\0",
                                                      _cat(proofs, 48) or b"\0", n, _sp(s)), "verify_cell_kzg_proof_batch")
    return bool(ok.value)


def verify_cell_kzg_proof_batches(batches: Sequence[Tuple[Sequence[bytes], Sequence[int], Sequence[bytes], Sequence[bytes]]], s) -> Tuple[List[bool], List[int]]:
    """K independent verify_cell_kzg_proof_batch checks in one call.  batches: (commitments, cell_indices, cells, proofs)
    per batch -> (verdict list, status list: the code the single call would return for each batch)."""
    k = len(batches)
    offsets = [0]
    for com, idx, cl, pr in batches:
        assert len(com) == len(idx) == len(cl) == len(pr)
        offsets.append(offsets[-1] + len(idx))
    n = offsets[-1]
    idx = (ctypes.c_uint64 * max(1, n))(*[i for b in batches for i in b[1]])
    off = _offsets(offsets)
    oks = (ctypes.c_bool * max(1, k))()
    st = _status_list(k)
    _check(load_library().lwkzg_verify_cell_kzg_proof_batches(oks, b"".join(_cat(b[0], 48) for b in batches) or b"\0", idx,
                                                              b"".join(_cat(b[2], BYTES_PER_CELL) for b in batches) or b"\0",
                                                              b"".join(_cat(b[3], 48) for b in batches) or b"\0", off, k, _sp(s), st),
           "lwkzg_verify_cell_kzg_proof_batches")
    return [bool(oks[i]) for i in range(k)], list(st)[:k]


def verify_cell_kzg_proof_batches_device(d_ok: int, d_commitments: int, d_cell_indices: int, d_cells: int, d_proofs: int, offsets: Sequence[int], s,
                                         stream: int = 0, d_status: int = 0):
    """All buffers are raw device addresses (torch: tensor.data_ptr()) except offsets (K + 1 host integers); d_ok and
    d_status are K int32 each.  Asynchronous on `stream`."""
    k = len(offsets) - 1
    off = _offsets(offsets)
    _check(load_library().lwkzg_verify_cell_kzg_proof_batches_device(d_ok or None, d_commitments or None, d_cell_indices or None, d_cells or None,
                                                                     d_proofs or None, off, k, _sp(s), stream or None, d_status or None),
           "lwkzg_verify_cell_kzg_proof_batches_device")


def verify_blob_cell_kzg_proof_batches(batches: Sequence[Tuple[Sequence[bytes], Sequence[bytes], Sequence[bytes]]], s) -> Tuple[List[bool], List[int]]:
    """K blob-transaction checks in one call.  batches: (blobs, commitments (one per blob), proofs (128 per blob,
    blob-major)) per batch -> (verdict list, status list): per batch, what compute_cells_and_kzg_proofs on its blobs
    followed by one verify_cell_kzg_proof_batch over all their cells gives."""
    k = len(batches)
    offsets = [0]
    for bl, com, pr in batches:
        assert len(bl) == len(com) and len(pr) == CELLS_PER_EXT_BLOB * len(bl)
        offsets.append(offsets[-1] + len(bl))
    off = _offsets(offsets)
    oks = (ctypes.c_bool * max(1, k))()
    st = _status_list(k)
    _check(load_library().lwkzg_verify_blob_cell_kzg_proof_batches(oks, b"".join(_cat(b[0], BYTES_PER_BLOB) for b in batches) or b"\0",
                                                                   b"".join(_cat(b[1], 48) for b in batches) or b"\0",
                                                                   b"".join(_cat(b[2], 48) for b in batches) or b"\0", off, k, _sp(s), st),
           "lwkzg_verify_blob_cell_kzg_proof_batches")
    return [bool(oks[i]) for i in range(k)], list(st)[:k]


def verify_blob_cell_kzg_proof_batches_device(d_ok: int, d_blobs: int, d_commitments: int, d_proofs: int, offsets: Sequence[int], s, stream: int = 0,
                                              d_status: int = 0):
    """All buffers are raw device addresses except offsets (K + 1 host integers, in blobs); d_ok and d_status are K
    int32 each.  Asynchronous on `stream`."""
    k = len(offsets) - 1
    off = _offsets(offsets)
    _check(load_library().lwkzg_verify_blob_cell_kzg_proof_batches_device(d_ok or None, d_blobs or None, d_commitments or None, d_proofs or None, off, k,
                                                                          _sp(s), stream or None, d_status or None),
           "lwkzg_verify_blob_cell_kzg_proof_batches_device")


def debug_cell_batch_challenges(n_batches: int, s) -> List[int]:
    """The challenges r_b the last verify_[blob_]cell_kzg_proof_batches[_device] call derived (0 for empty batches; test hook)."""
    return _debug_challenges("lwkzg_debug_cell_batch_challenges", n_batches, s)


def cell_window_bits(s) -> int:
    return int(load_library().lwkzg_cell_window_bits(_sp(s)))


def debug_cell_stages(blob: bytes, s):
    """-> (scalars [j][b] as ints, Hhat_j compressed, H positions compressed, FK20 points as (x, y) ints or None)."""
    sc = ctypes.create_string_buffer(8192 * 32)
    hh = ctypes.create_string_buffer(128 * 48)
    h = ctypes.create_string_buffer(128 * 48)
    fk = ctypes.create_string_buffer(8192 * 96)
    _check(load_library().lwkzg_debug_cell_stages(sc, hh, h, fk, blob, _sp(s)), "lwkzg_debug_cell_stages")
    # the library's MSM order is (j // 64) * 4096 + b * 64 + j % 64; returned here as [j * 64 + b]
    order = [(j // 64) * 4096 + b * 64 + j % 64 for j in range(128) for b in range(64)]
    scalars = [int.from_bytes(sc.raw[32 * i: 32 * i + 32], "little") for i in order]
    pts = []
    for i in order:
        x = int.from_bytes(fk.raw[96 * i: 96 * i + 48], "little")
        y = int.from_bytes(fk.raw[96 * i + 48: 96 * i + 96], "little")
        pts.append(None if x == 0 and y == 0 else (x, y))
    return scalars, [hh.raw[48 * i: 48 * i + 48] for i in range(128)], [h.raw[48 * i: 48 * i + 48] for i in range(128)], pts


def table_share(s) -> int:
    """0 = private digit table, 1 = built here and published, 2 = attached to another process's, 3 = shared in-process."""
    return int(load_library().lwkzg_table_share(_sp(s)))
