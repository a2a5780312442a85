"""GPU tier: many independent cell-proof batches per call, lwkzg_verify_cell_kzg_proof_batches[_device] (include/lwkzg.h
part 3).

Every batch must get exactly what one verify_cell_kzg_proof_batch call on it alone gives (verdict and error code), its
challenge must be the oracle's, and a forged pair that only the batch's random weights catch must fail its own batch
and no other."""
import ctypes
import os

import pytest

from tests import _forge
from tests.golden.make_cell_fixtures import make_blob

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
R = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
NBLOBS = 12


@pytest.fixture(scope="module")
def lw():
    import lambdaworks_kzg_b200 as m

    m.load_library()
    return m


def _load(lw, mode):
    lw.set_option("mode", mode)
    lw.set_option("window_bits", 8)
    lw.set_option("cell_window_bits", 8)
    try:
        return lw.load_trusted_setup_file(os.path.join(GOLDEN, "trusted_setup.txt"))
    finally:
        lw.set_option("mode", 0)
        lw.set_option("window_bits", 13)
        lw.set_option("cell_window_bits", 13)


class Data:
    """NBLOBS blobs of one mode: commitments, and every cell and proof from the compute batch."""

    def __init__(self, lw, s, mode):
        self.s, self.mode = s, mode
        blobs = b"".join(make_blob(300 + b, mode) for b in range(NBLOBS))
        self.coms, st = lw.blob_to_kzg_commitment_batch(blobs, NBLOBS, s)
        assert st == [0] * NBLOBS
        cells, proofs, st = lw.compute_cells_and_kzg_proofs_batch(blobs, NBLOBS, s)
        assert st == [0] * NBLOBS
        self.cells, self.proofs = cells, proofs

    def cell(self, b, k):
        return self.cells[(b * 128 + k) * 2048: (b * 128 + k + 1) * 2048]

    def proof(self, b, k):
        return self.proofs[(b * 128 + k) * 48: (b * 128 + k + 1) * 48]

    def batch(self, sel):
        """[(blob, cell index)] -> (commitments, indices, cells, proofs)"""
        return ([self.coms[b] for b, _ in sel], [k for _, k in sel], [self.cell(b, k) for b, k in sel], [self.proof(b, k) for b, k in sel])


@pytest.fixture(scope="module", params=[2, 0, 1], ids=["mode2", "mode0", "mode1"])
def data(request, lw):
    s = _load(lw, request.param)
    yield Data(lw, s, request.param)
    s.free()


@pytest.fixture(scope="module")
def d2(lw):
    s = _load(lw, 2)
    yield Data(lw, s, 2)
    s.free()


def _single(lw, batch, s):
    """(ok, code) of one verify_cell_kzg_proof_batch call"""
    try:
        return lw.verify_cell_kzg_proof_batch(*batch, s), 0
    except lw.KzgError as e:
        return False, e.code


def _mixed(d):
    """the PeerDAS shape (one batch per column over NBLOBS blobs) among small, empty, large and bad batches"""
    out = [d.batch([])]
    out += [d.batch([(b, col) for b in range(NBLOBS)]) for col in range(128)]
    out.append(d.batch([(4, 77)]))
    out.append(d.batch([]))
    out.append(d.batch([(0, 3), (1, 9), (0, 70), (2, 5), (1, 100), (0, 3)]))        # repeated commitments, mixed indices
    out.append(d.batch([(b, k) for b in range(5) for k in range(120)]))             # 600 cells
    out.append(d.batch([(3, 1), (4, 1), (5, 1)]))
    c, i, cl, p = d.batch([(3, 1), (4, 1), (5, 1)])
    out.append((c, i, cl, [p[1], p[0], p[2]]))                                      # swapped proofs
    c, i, cl, p = d.batch([(6, 10), (6, 11), (7, 12)])
    out.append((c, i, [cl[0], d.cell(6, 12), cl[2]], p))                            # wrong cell
    c, i, cl, p = d.batch([(8, 20), (9, 21)])
    out.append(([c[0], d.coms[10]], i, cl, p))                                      # wrong commitment
    out.append(d.batch([(11, 127), (10, 0)]))
    out.append(d.batch([]))
    return out


def _dedup(coms):
    uniq, cidx = [], []
    for c in coms:
        if c not in uniq:
            uniq.append(c)
        cidx.append(uniq.index(c))
    return uniq, cidx


def test_agreement_with_single_calls(lw, data, py_setup):
    from oracle.py import cells as ocells

    batches = _mixed(data)
    oks, sts = lw.verify_cell_kzg_proof_batches(batches, data.s)
    want = [_single(lw, b, data.s) for b in batches]
    assert oks == [w[0] for w in want] and sts == [w[1] for w in want]
    assert sts == [0] * len(batches)
    assert oks[:130] == [True] * 130 and oks[-8:] == [True, True, True, False, False, False, True, True]
    # the challenges of every non-empty batch (including the one with repeated commitments) against the oracle
    o = ocells.CellOracle(py_setup, data.mode)
    rs = lw.debug_cell_batch_challenges(len(batches), data.s)
    for b, (c, i, cl, p) in enumerate(batches):
        if not i:
            assert rs[b] == 0, b
            continue
        if b in range(1, 129, 9) or b >= 129:
            uniq, cidx = _dedup(c)
            assert rs[b] == o.batch_challenge(uniq, cidx, i, cl, p), b
    # the oracle's verdict on a sample
    for b in (129, 131, 133, 134, 135, 136):
        assert o.verify_cell_kzg_proof_batch(*batches[b]) is oks[b], b


def _forged(d, tau, sel, i, j):
    c, idx, cl, p = d.batch(sel)
    return (c, idx, cl, _forge.forge_cell_batch(tau, idx, p, i, j))


def test_forged_pairs(lw, d2, py_setup):
    """Forged pairs pass exactly when their two weights are equal: at local (0, 1), (i, i + 32), (i, i + 64), in a batch
    after a pass boundary, and at the first cell of a later batch."""
    from oracle.py import cells as ocells

    o = ocells.CellOracle(py_setup, 2)
    tau = py_setup.tau
    good = d2.batch([(b, 40) for b in range(NBLOBS)])
    big = [(b % NBLOBS, (b * 7) % 128) for b in range(100)]
    cases = [
        [good, _forged(d2, tau, [(b, 40) for b in range(NBLOBS)], 0, 1), good],
        [good, good, _forged(d2, tau, big, 3, 35), good],
        [good, _forged(d2, tau, big, 5, 69), good],
        [good, d2.batch([]), _forged(d2, tau, [(b, 9) for b in range(NBLOBS)] + [(0, 5)], 0, 12)],
    ]
    for bi, batches in enumerate(cases):
        forged_at = [k for k, b in enumerate(batches) if b is not good and b[1]][0]
        oks, sts = lw.verify_cell_kzg_proof_batches(batches, d2.s)
        assert sts == [0] * len(batches)
        assert oks == [k != forged_at for k in range(len(batches))], bi
        assert o.verify_cell_kzg_proof_batch(*batches[forged_at]) is False
        assert _forge.weighted_cell_check(o, *batches[forged_at], [1] * len(batches[forged_at][1])) is True
    # across a pass boundary: passes of at most 128 cells put each 100-cell batch in a pass of its own
    lw.set_option("cell_chunk_blobs", 1)
    try:
        batches = [d2.batch(big), d2.batch(big[:50]), _forged(d2, tau, big, 0, 64), d2.batch(big)]
        oks, sts = lw.verify_cell_kzg_proof_batches(batches, d2.s)
    finally:
        lw.set_option("cell_chunk_blobs", 888)
    assert sts == [0] * 4 and oks == [True, True, False, True]


def test_points_outside_g1(lw, d2):
    good = d2.batch([(b, 3) for b in range(4)])
    for enc in _forge.non_g1_points():
        c, i, cl, p = good
        bad_proof = (c, i, cl, [p[0], enc] + p[2:])
        bad_com = ([c[0], c[1], enc, c[3]], i, cl, p)
        oks, sts = lw.verify_cell_kzg_proof_batches([good, bad_proof, good, bad_com, good], d2.s)
        assert sts == [0, lw.C_KZG_BADARGS, 0, lw.C_KZG_BADARGS, 0] and oks == [True, False, True, False, True]
        oks, sts = lw.verify_cell_kzg_proof_batches([good, good], d2.s)
        assert oks == [True, True] and sts == [0, 0]


def _raw(lw, batches, s, status=True):
    k = len(batches)
    offs = [0]
    for b in batches:
        offs.append(offs[-1] + len(b[1]))
    n = offs[-1]
    ok = (ctypes.c_bool * k)(*([True] * k))
    st = (ctypes.c_int * k)(*([-7] * k)) if status else None
    idx = (ctypes.c_uint64 * max(1, n))(*[i for b in batches for i in b[1]])
    code = lw.load_library().lwkzg_verify_cell_kzg_proof_batches(ok, b"".join(c for b in batches for c in b[0]), idx,
                                                                 b"".join(c for b in batches for c in b[2]), b"".join(c for b in batches for c in b[3]),
                                                                 (ctypes.c_uint64 * (k + 1))(*offs), k, s.ptr, st)
    return code, list(ok), (list(st) if status else None)


@pytest.mark.parametrize("mode", [2, 0])
def test_per_batch_errors(lw, d2, mode):
    d = d2 if mode == 2 else Data(lw, _load(lw, 0), 0)
    try:
        code = lw.C_KZG_BADARGS if mode == 2 else lw.C_KZG_ERROR
        good = d.batch([(b, 17) for b in range(6)])
        c, i, cl, p = good
        bad_index = (c, i[:2] + [128] + i[3:], cl, p)
        bad_word = (c, i, cl[:1] + [cl[1][:64] + R.to_bytes(32, "big") + cl[1][96:]] + cl[2:], p)
        bad_proof = (c, i, cl, p[:4] + [b"\x9f" + b"\xff" * 47] + p[5:])   # x >= p
        for bad in (bad_index, bad_word, bad_proof):
            batches = [good, good, bad, good]
            want_ok, want_code = _single(lw, bad, d.s)
            assert not want_ok and (want_code == code or bad is bad_proof)
            oks, sts = lw.verify_cell_kzg_proof_batches(batches, d.s)
            assert sts == [0, 0, want_code, 0] and oks == [True, True, False, True]
            rc, ok, _ = _raw(lw, batches, d.s, status=False)
            assert rc == want_code and ok == [True, True, False, True]
    finally:
        if d is not d2:
            d.s.free()


def test_whole_call_errors(lw, d2):
    lib = lw.load_library()
    c, i, cl, p = d2.batch([(0, 1), (1, 2)])
    com, cells, prf = b"".join(c), b"".join(cl), b"".join(p)
    idx = (ctypes.c_uint64 * 2)(*i)
    ok = (ctypes.c_bool * 2)(True, True)
    st = (ctypes.c_int * 2)(-7, -7)
    f = lib.lwkzg_verify_cell_kzg_proof_batches
    U = ctypes.c_uint64
    # n_batches == 0: OK, nothing written
    assert f(ok, com, idx, cells, prf, (U * 1)(0), 0, d2.s.ptr, st) == lw.C_KZG_OK and list(st) == [-7, -7]
    assert f(None, com, idx, cells, prf, (U * 2)(0, 2), 1, d2.s.ptr, st) == lw.C_KZG_BADARGS
    assert f(ok, com, idx, cells, prf, None, 1, d2.s.ptr, st) == lw.C_KZG_BADARGS
    for k in range(4):
        args = [com, idx, cells, prf]
        args[k] = None
        assert f(ok, *args, (U * 2)(0, 2), 1, d2.s.ptr, st) == lw.C_KZG_BADARGS
    assert f(ok, com, idx, cells, prf, (U * 2)(1, 2), 1, d2.s.ptr, st) == lw.C_KZG_BADARGS
    assert f(ok, com, idx, cells, prf, (U * 3)(0, 2, 1), 2, d2.s.ptr, st) == lw.C_KZG_BADARGS
    assert f(ok, com, idx, cells, prf, (U * 2)(0, (1 << 24) + 1), 1, d2.s.ptr, st) == lw.C_KZG_BADARGS
    assert list(st) == [-7, -7]
    # only empty batches: nothing to read
    assert f(ok, None, None, None, None, (U * 3)(0, 0, 0), 2, d2.s.ptr, st) == lw.C_KZG_OK and list(ok) == [True, True] and list(st) == [0, 0]
    g = lib.lwkzg_verify_cell_kzg_proof_batches_device
    assert g(None, 1 << 20, 1 << 20, 1 << 20, 1 << 20, (U * 2)(0, 2), 1, d2.s.ptr, None, None) == lw.C_KZG_BADARGS
    assert g(1 << 20, 1 << 20, 1 << 20, 1 << 20, 1 << 20, (U * 2)(3, 2), 1, d2.s.ptr, None, None) == lw.C_KZG_BADARGS
    assert g(1 << 20, 1 << 20, 1 << 20, 1 << 20, 1 << 20, None, 0, d2.s.ptr, None, None) == lw.C_KZG_OK


def _device(lw, torch, batches, s, with_status=True, stream=None, producer=False):
    offs = [0]
    for b in batches:
        offs.append(offs[-1] + len(b[1]))
    k = len(batches)

    def dev(raw, dtype=torch.uint8):
        return torch.frombuffer(bytearray(raw or b"\0" * 16), dtype=dtype).cuda()

    d_c = dev(b"".join(c for b in batches for c in b[0]))
    d_i = torch.tensor([i for b in batches for i in b[1]] or [0], dtype=torch.int64, device="cuda")
    d_src = dev(b"".join(c for b in batches for c in b[2]))
    d_p = dev(b"".join(c for b in batches for c in b[3]))
    d_ok = torch.full((k,), -7, dtype=torch.int32, device="cuda")
    d_st = torch.full((k,), -7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    st = stream or torch.cuda.current_stream()
    with torch.cuda.stream(st):
        d_cells = torch.add(d_src, 0) if producer else d_src   # written by a kernel on `st` right before the call
        lw.verify_cell_kzg_proof_batches_device(d_ok.data_ptr(), d_c.data_ptr(), d_i.data_ptr(), d_cells.data_ptr(), d_p.data_ptr(), offs, s,
                                                st.cuda_stream, d_st.data_ptr() if with_status else 0)
        oks, sts = d_ok.cpu().tolist(), d_st.cpu().tolist()
    torch.cuda.synchronize()
    return [bool(v) for v in oks], sts


def test_device_form(lw, d2):
    import torch

    batches = _mixed(d2)
    c, i, cl, p = d2.batch([(b, 17) for b in range(6)])
    batches.insert(5, (c, i[:2] + [128] + i[3:], cl, p))
    batches.insert(9, (c, i, cl, p[:4] + [b"\xff" * 48] + p[5:]))
    oks, sts = lw.verify_cell_kzg_proof_batches(batches, d2.s)
    assert sts[5] == sts[9] == lw.C_KZG_BADARGS and not oks[5] and not oks[9]
    rs = lw.debug_cell_batch_challenges(len(batches), d2.s)
    d_oks, d_sts = _device(lw, torch, batches, d2.s)
    assert d_oks == oks and d_sts == sts
    assert lw.debug_cell_batch_challenges(len(batches), d2.s) == rs
    d_oks, d_sts = _device(lw, torch, batches, d2.s, with_status=False)
    assert d_oks == oks and d_sts == [-7] * len(batches)
    d_oks, d_sts = _device(lw, torch, batches, d2.s, stream=torch.cuda.Stream(), producer=True)
    assert d_oks == oks and d_sts == sts
    # several passes (at most 2 x 128 cells each: the 600-cell batch alone) give the same verdicts and challenges
    lw.set_option("cell_chunk_blobs", 2)
    try:
        d_oks, d_sts = _device(lw, torch, batches, d2.s)
        assert lw.debug_cell_batch_challenges(len(batches), d2.s) == rs
        h_oks, h_sts = lw.verify_cell_kzg_proof_batches(batches, d2.s)
    finally:
        lw.set_option("cell_chunk_blobs", 888)
    assert d_oks == h_oks == oks and d_sts == h_sts == sts
    assert lw.debug_cell_batch_challenges(len(batches), d2.s) == rs


def test_settings_without_monomial_srs(lw, d2):
    """Hand-built settings in a Lagrange mode carry no monomial SRS: a call with cells fails as the single call does
    (C_KZG_ERROR), a call of empty batches only verifies, as the single call with no cells does."""
    import torch
    from lambdaworks_kzg_b200.api import CKZGSettings

    g1 = ctypes.create_string_buffer(d2.s.g1_values_bytes(), 4096 * 144)
    g2 = ctypes.create_string_buffer(d2.s.g2_values_bytes(), 65 * 288)
    lw.set_option("mode", 2)
    lw.set_option("window_bits", 8)
    try:
        s = CKZGSettings(None, ctypes.cast(g1, ctypes.c_void_p), ctypes.cast(g2, ctypes.c_void_p))
        batch = d2.batch([(0, 1), (1, 2)])
        ok1, code = _single(lw, batch, s)
        assert not ok1 and code == lw.C_KZG_ERROR
        with pytest.raises(lw.KzgError) as e:
            lw.verify_cell_kzg_proof_batches([d2.batch([]), batch], s)
        assert e.value.code == code
        assert _single(lw, d2.batch([]), s) == (True, 0)
        assert lw.verify_cell_kzg_proof_batches([d2.batch([]), d2.batch([])], s) == ([True, True], [0, 0])
        d_ok = torch.full((2,), -7, dtype=torch.int32, device="cuda")
        d_st = torch.full((2,), -7, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        lw.verify_cell_kzg_proof_batches_device(d_ok.data_ptr(), 0, 0, 0, 0, [0, 0, 0], s, torch.cuda.current_stream().cuda_stream, d_st.data_ptr())
        torch.cuda.synchronize()
        assert d_ok.tolist() == [1, 1] and d_st.tolist() == [0, 0]
        with pytest.raises(lw.KzgError) as e:
            lw.verify_cell_kzg_proof_batches_device(d_ok.data_ptr(), 1 << 20, 1 << 20, 1 << 20, 1 << 20, [0, 2], s)
        assert e.value.code == code
    finally:
        lw.set_option("mode", 0)
        lw.set_option("window_bits", 13)
