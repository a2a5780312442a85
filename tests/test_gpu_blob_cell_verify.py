"""GPU tier: cell-proof verification straight from blobs, lwkzg_verify_blob_cell_kzg_proof_batches[_device]
(include/lwkzg.h part 3).

Every batch must get exactly what the composition it replaces gives: compute_cells_and_kzg_proofs on each of its blobs
(a failure is the batch's verdict and code), then one verify_cell_kzg_proof_batch over their cells with each blob's
commitment repeated 128 times and cell indices 0..127 -- here lwkzg_verify_cell_kzg_proof_batches on those composed
inputs, which also gives the challenge r_b each batch must share."""
import ctypes
import os

import pytest

from tests import _forge
from tests.golden.make_cell_fixtures import make_blob

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
R = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
NBLOBS = 8


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
    """NBLOBS blobs of one mode with their commitments and 128 proofs each."""

    def __init__(self, lw, s, mode):
        self.s, self.mode = s, mode
        self.blobs = [make_blob(700 + b, mode) for b in range(NBLOBS)]
        self.coms, st = lw.blob_to_kzg_commitment_batch(b"".join(self.blobs), NBLOBS, s)
        assert st == [0] * NBLOBS
        _, proofs, st = lw.compute_cells_and_kzg_proofs_batch(b"".join(self.blobs), NBLOBS, s, want_cells=False)
        assert st == [0] * NBLOBS
        self.proofs = [[proofs[(b * 128 + k) * 48: (b * 128 + k + 1) * 48] for k in range(128)] for b in range(NBLOBS)]

    def tx(self, sel):
        """[blob] -> (blobs, commitments, proofs): a transaction as the network wrapper carries it"""
        return [self.blobs[b] for b in sel], [self.coms[b] for b in sel], [p for b in sel for p in self.proofs[b]]


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


def _composed_inputs(lw, batches, s):
    """-> (cell batches, compute codes): the cells of every blob from lwkzg_compute_cells_and_kzg_proofs_batch, each
    batch as (commitments x 128, indices 0..127, cells, proofs); the first failing blob's code per batch (0 if none)"""
    flat = [bl for b in batches for bl in b[0]]
    cells, _, st = lw.compute_cells_and_kzg_proofs_batch(b"".join(flat), len(flat), s, want_proofs=False) if flat else (b"", b"", [])
    out, codes, at = [], [], 0
    for bl, com, pr in batches:
        n = len(bl)
        codes.append(next((c for c in st[at: at + n] if c), 0))
        cl = [cells[((at + i) * 128 + k) * 2048: ((at + i) * 128 + k + 1) * 2048] for i in range(n) for k in range(128)]
        out.append(([c for c in com for _ in range(128)], [k for _ in range(n) for k in range(128)], cl, list(pr)))
        at += n
    return out, codes


def _composed(lw, batches, s):
    """(oks, statuses, challenges) of the composition; challenges are None for batches whose cells could not be computed"""
    cb, codes = _composed_inputs(lw, batches, s)
    runnable = [b if code == 0 else ([], [], [], []) for b, code in zip(cb, codes)]
    oks, sts = lw.verify_cell_kzg_proof_batches(runnable, s)
    rs = lw.debug_cell_batch_challenges(len(batches), s)
    for i, code in enumerate(codes):
        if code:
            oks[i], sts[i], rs[i] = False, code, None
    return oks, sts, rs


def _new(lw, batches, s):
    oks, sts = lw.verify_blob_cell_kzg_proof_batches(batches, s)
    return oks, sts, lw.debug_cell_batch_challenges(len(batches), s)


def _same(got, want):
    g_ok, g_st, g_rs = got
    w_ok, w_st, w_rs = want
    assert g_ok == w_ok and g_st == w_st
    for b, r in enumerate(w_rs):
        if r is not None:
            assert g_rs[b] == r, b


def _set_word(d, blob, i, raw):
    return blob[:32 * i] + raw + blob[32 * i + 32:]


def _mixed(d):
    """transactions of 0, 1, 2 and 6 blobs, valid and not"""
    out = [d.tx([])]
    out.append(d.tx([0]))
    out.append(d.tx([0, 1, 2, 3, 4, 5]))
    out.append(d.tx([]))
    out.append(d.tx([2, 2]))                                                        # one blob twice under one commitment
    bl, com, pr = d.tx([3, 4])
    out.append((bl, [com[1], com[0]], pr))                                          # swapped commitments
    bl, com, pr = d.tx([5, 6])
    out.append((bl, com, pr[:128 + 40] + [d.proofs[0][40]] + pr[128 + 41:]))        # one wrong proof
    out.append(([d.blobs[1]], [d.coms[1]], d.proofs[7]))                            # blob 7's proofs attached to blob 1
    out.append(([d.blobs[4]], [d.coms[4]], d.proofs[4][1:] + d.proofs[4][:1]))      # proofs shifted by one cell
    out.append(([_set_word(d, d.blobs[3], 100, _forge.fe_bytes(d.mode, 12345))], [d.coms[3]], d.proofs[3]))   # blob changed, rest kept
    out.append(d.tx([2, 3, 4, 5, 6, 7]))
    out.append(d.tx([7]))
    out.append(d.tx([]))
    return out


MIXED_OK = [True, True, True, True, True, False, False, False, False, False, True, True, True]


def test_agreement_with_composition(lw, data, py_setup):
    from oracle.py import cells as ocells

    batches = _mixed(data)
    want = _composed(lw, batches, data.s)
    got = _new(lw, batches, data.s)
    _same(got, want)
    assert got[0] == MIXED_OK and got[1] == [0] * len(batches)
    assert all(r != 0 for b, r in zip(batches, got[2]) if b[0]) and all(r == 0 for b, r in zip(batches, got[2]) if not b[0])
    # a sample against the oracle: the challenge with a repeated commitment, and two verdicts
    o = ocells.CellOracle(py_setup, data.mode)
    cb, _ = _composed_inputs(lw, batches, data.s)
    c, i, cl, p = cb[4]
    assert got[2][4] == o.batch_challenge([c[0]], [0] * len(i), i, cl, p)
    for b in (1, 8):
        assert o.verify_cell_kzg_proof_batch(*cb[b]) is got[0][b], b


def test_per_batch_failures(lw, data):
    """A blob word >= r (modes 1 and 2), a commitment or proof that does not decode, and points outside G1 fail their own
    batch only, with the composed path's code."""
    code = lw.C_KZG_ERROR if data.mode == 0 else lw.C_KZG_BADARGS
    good = data.tx([0, 1])
    bl, com, pr = good
    bad = [
        (bl, [com[0], b"\x9f" + b"\xff" * 47], pr),                                 # commitment x >= p
        (bl, com, pr[:130] + [b"\xff" * 48] + pr[131:]),                            # proof that does not decode
    ]
    for enc in _forge.non_g1_points():
        bad.append((bl, [enc, com[1]], pr))
        bad.append((bl, com, pr[:7] + [enc] + pr[8:]))
    if data.mode != 0:
        # a word >= r whose reduction is an ordinary field element: only the blob check can reject it
        bad.append(([bl[0], _set_word(data, bl[1], 4000, (R + 12345).to_bytes(32, "little" if data.mode == 1 else "big"))], com, pr))
    for x in bad:
        batches = [good, data.tx([]), x, good]
        want = _composed(lw, batches, data.s)
        got = _new(lw, batches, data.s)
        _same(got, want)
        want_code = want[1][2]
        assert want_code == code or (data.mode == 0 and want_code == 0)   # MODE_REFERENCE's decoder accepts some encodings
        assert got[1] == [0, 0, want_code, 0] and [got[0][k] for k in (0, 1, 3)] == [True, True, True]
        k = len(batches)
        ok = (ctypes.c_bool * k)(*([True] * k))
        rc = _raw(lw, batches, data.s, ok, None)
        assert rc == want_code and list(ok) == got[0]
        if want_code:
            assert not got[0][2]


def _forged(d, tau, sel, blob_pos, i, j):
    """transaction sel with blob sel[blob_pos]'s proofs forged at its cells (i, j)"""
    bl, com, pr = d.tx(sel)
    idx = [k for _ in sel for k in range(128)]
    return bl, com, _forge.forge_cell_batch(tau, idx, pr, 128 * blob_pos + i, 128 * blob_pos + j)


def test_forged_pairs(lw, d2, py_setup):
    """Forged pairs only the batch's random weights catch: at cells (0, 1), (i, i + 32), (i, i + 64) of one blob, and in
    a batch after a pass boundary.  The forged batch fails, its neighbours pass, and unit weights accept it."""
    from oracle.py import cells as ocells

    o = ocells.CellOracle(py_setup, 2)
    tau = py_setup.tau
    good = d2.tx([0, 1])
    cases = [   # (batches, index of the forged one)
        ([good, _forged(d2, tau, [2], 0, 0, 1), good], 1),
        ([good, good, _forged(d2, tau, [3, 4], 1, 5, 37), good], 2),
        ([good, _forged(d2, tau, [5], 0, 20, 84), d2.tx([6])], 1),
    ]
    for batches, at in cases:
        oks, sts = lw.verify_blob_cell_kzg_proof_batches(batches, d2.s)
        assert sts == [0] * len(batches)
        assert oks == [k != at for k in range(len(batches))], at
        cb, _ = _composed_inputs(lw, batches[at: at + 1], d2.s)
        assert _forge.weighted_cell_check(o, *cb[0], [1] * len(cb[0][1])) is True
    # passes of at most one blob: the 2-blob batches get a pass each, the forged batch follows a pass boundary
    lw.set_option("cell_chunk_blobs", 1)
    try:
        batches = [d2.tx([0]), good, _forged(d2, tau, [7], 0, 9, 73), d2.tx([6]), d2.tx([3, 4])]
        oks, sts = lw.verify_blob_cell_kzg_proof_batches(batches, d2.s)
    finally:
        lw.set_option("cell_chunk_blobs", 888)
    assert sts == [0] * 5 and oks == [True, True, False, True, True]
    cb, _ = _composed_inputs(lw, batches[2:3], d2.s)
    assert _forge.weighted_cell_check(o, *cb[0], [1] * 128) is True


def _raw(lw, batches, s, ok, st):
    offs = [0]
    for b in batches:
        offs.append(offs[-1] + len(b[0]))
    k = len(offs) - 1
    return lw.load_library().lwkzg_verify_blob_cell_kzg_proof_batches(ok, b"".join(x for b in batches for x in b[0]) or b"\0",
                                                                      b"".join(x for b in batches for x in b[1]) or b"\0",
                                                                      b"".join(x for b in batches for x in b[2]) or b"\0",
                                                                      (ctypes.c_uint64 * (k + 1))(*offs), k, s.ptr, st)


def test_whole_call_errors(lw, d2):
    lib = lw.load_library()
    bl, com, pr = d2.tx([0, 1])
    blobs, coms, prf = b"".join(bl), b"".join(com), b"".join(pr)
    ok = (ctypes.c_bool * 2)(True, True)
    st = (ctypes.c_int * 2)(-7, -7)
    f = lib.lwkzg_verify_blob_cell_kzg_proof_batches
    U = ctypes.c_uint64
    # n_batches == 0: OK, nothing written
    assert f(ok, blobs, coms, prf, (U * 1)(0), 0, d2.s.ptr, st) == lw.C_KZG_OK and list(st) == [-7, -7]
    assert f(None, blobs, coms, prf, (U * 2)(0, 2), 1, d2.s.ptr, st) == lw.C_KZG_BADARGS
    assert f(ok, blobs, coms, prf, None, 1, d2.s.ptr, st) == lw.C_KZG_BADARGS
    for k in range(3):
        args = [blobs, coms, prf]
        args[k] = None
        assert f(ok, *args, (U * 2)(0, 2), 1, d2.s.ptr, st) == lw.C_KZG_BADARGS
    assert f(ok, blobs, coms, prf, (U * 2)(1, 2), 1, d2.s.ptr, st) == lw.C_KZG_BADARGS
    assert f(ok, blobs, coms, prf, (U * 3)(0, 2, 1), 2, d2.s.ptr, st) == lw.C_KZG_BADARGS
    # more than 2^24 cells, and a count whose cells overflow 64 bits, are rejected before any input is read
    tiny = b"\0" * 16
    assert f(ok, tiny, tiny, tiny, (U * 2)(0, (1 << 17) + 1), 1, d2.s.ptr, st) == lw.C_KZG_BADARGS
    assert f(ok, tiny, tiny, tiny, (U * 3)(0, 1, 1 << 57), 2, d2.s.ptr, st) == lw.C_KZG_BADARGS
    assert list(st) == [-7, -7] and list(ok) == [True, True]
    # only empty batches: nothing to read
    assert f(ok, None, None, None, (U * 3)(0, 0, 0), 2, d2.s.ptr, st) == lw.C_KZG_OK and list(ok) == [True, True] and list(st) == [0, 0]
    # with status == NULL the first failing batch's code is returned and ok is still filled
    ok3 = (ctypes.c_bool * 3)(False, True, False)
    bad = (bl, [com[0], b"\xff" * 48], pr)
    assert _raw(lw, [d2.tx([0]), bad, d2.tx([1])], d2.s, ok3, None) == lw.C_KZG_BADARGS and list(ok3) == [True, False, True]
    g = lib.lwkzg_verify_blob_cell_kzg_proof_batches_device
    assert g(None, 1 << 20, 1 << 20, 1 << 20, (U * 2)(0, 2), 1, d2.s.ptr, None, None) == lw.C_KZG_BADARGS
    assert g(1 << 20, 1 << 20, 1 << 20, 1 << 20, (U * 2)(3, 2), 1, d2.s.ptr, None, None) == lw.C_KZG_BADARGS
    assert g(1 << 20, 1 << 20, 1 << 20, None, (U * 2)(0, 2), 1, d2.s.ptr, None, None) == lw.C_KZG_BADARGS
    assert g(1 << 20, 1 << 20, 1 << 20, 1 << 20, (U * 2)(0, (1 << 17) + 1), 1, d2.s.ptr, None, None) == lw.C_KZG_BADARGS
    assert g(1 << 20, 1 << 20, 1 << 20, 1 << 20, None, 0, d2.s.ptr, None, None) == lw.C_KZG_OK


def test_settings_without_monomial_srs(lw, d2):
    """Hand-built settings in a Lagrange mode carry no monomial SRS: a call with blobs fails with C_KZG_ERROR, a call of
    empty batches only verifies."""
    import torch
    from lambdaworks_kzg_b200.api import CKZGSettings

    g1 = ctypes.create_string_buffer(d2.s.g1_values_bytes(), 4096 * 144)
    g2 = ctypes.create_string_buffer(d2.s.g2_values_bytes(), 65 * 288)
    lw.set_option("mode", 2)
    lw.set_option("window_bits", 8)
    try:
        s = CKZGSettings(None, ctypes.cast(g1, ctypes.c_void_p), ctypes.cast(g2, ctypes.c_void_p))
        with pytest.raises(lw.KzgError) as e:
            lw.verify_blob_cell_kzg_proof_batches([d2.tx([]), d2.tx([0])], s)
        assert e.value.code == lw.C_KZG_ERROR
        assert lw.verify_blob_cell_kzg_proof_batches([d2.tx([]), d2.tx([])], s) == ([True, True], [0, 0])
        d_ok = torch.full((2,), -7, dtype=torch.int32, device="cuda")
        d_st = torch.full((2,), -7, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        lw.verify_blob_cell_kzg_proof_batches_device(d_ok.data_ptr(), 0, 0, 0, [0, 0, 0], s, torch.cuda.current_stream().cuda_stream, d_st.data_ptr())
        torch.cuda.synchronize()
        assert d_ok.tolist() == [1, 1] and d_st.tolist() == [0, 0]
        with pytest.raises(lw.KzgError) as e:
            lw.verify_blob_cell_kzg_proof_batches_device(d_ok.data_ptr(), 1 << 20, 1 << 20, 1 << 20, [0, 2], s)
        assert e.value.code == lw.C_KZG_ERROR
    finally:
        lw.set_option("mode", 0)
        lw.set_option("window_bits", 13)


def _device(lw, torch, batches, s, with_status=True, stream=None, producer=False):
    offs = [0]
    for b in batches:
        offs.append(offs[-1] + len(b[0]))
    k = len(batches)

    def dev(raw):
        return torch.frombuffer(bytearray(raw or b"\0" * 16), dtype=torch.uint8).cuda()

    d_src = dev(b"".join(x for b in batches for x in b[0]))
    d_c = dev(b"".join(x for b in batches for x in b[1]))
    d_p = dev(b"".join(x for b in batches for x in b[2]))
    d_ok = torch.full((k,), -7, dtype=torch.int32, device="cuda")
    d_st = torch.full((k,), -7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    st = stream or torch.cuda.current_stream()
    with torch.cuda.stream(st):
        d_b = torch.add(d_src, 0) if producer else d_src   # written by a kernel on `st` right before the call
        lw.verify_blob_cell_kzg_proof_batches_device(d_ok.data_ptr(), d_b.data_ptr(), d_c.data_ptr(), d_p.data_ptr(), offs, s, st.cuda_stream,
                                                     d_st.data_ptr() if with_status else 0)
        oks, sts = d_ok.cpu().tolist(), d_st.cpu().tolist()
    torch.cuda.synchronize()
    return [bool(v) for v in oks], sts


def test_device_form(lw, d2):
    import torch

    batches = _mixed(d2)
    bl, com, pr = d2.tx([0, 1])
    batches.insert(5, ([bl[0], _set_word(d2, bl[1], 7, b"\xff" * 32)], com, pr))
    batches.insert(9, (bl, com, pr[:4] + [b"\xff" * 48] + pr[5:]))
    oks, sts, rs = _new(lw, batches, d2.s)
    assert sts[5] == sts[9] == lw.C_KZG_BADARGS and not oks[5] and not oks[9]
    assert oks == MIXED_OK[:5] + [False] + MIXED_OK[5:8] + [False] + MIXED_OK[8:]
    assert _device(lw, torch, batches, d2.s) == (oks, sts)
    assert lw.debug_cell_batch_challenges(len(batches), d2.s) == rs
    assert _device(lw, torch, batches, d2.s, with_status=False) == (oks, [-7] * len(batches))
    assert _device(lw, torch, batches, d2.s, stream=torch.cuda.Stream(), producer=True) == (oks, sts)
    # several passes of at most 2 blobs (the 6-blob batches alone, larger than a pass), host and device alike
    lw.set_option("cell_chunk_blobs", 2)
    try:
        d_res = _device(lw, torch, batches, d2.s)
        assert lw.debug_cell_batch_challenges(len(batches), d2.s) == rs
        h_res = _new(lw, batches, d2.s)
    finally:
        lw.set_option("cell_chunk_blobs", 888)
    assert d_res == (oks, sts) and h_res == (oks, sts, rs)


def test_extension_in_sub_passes(lw, d2):
    """Fresh settings whose first cell call is this one with passes of at most 2 blobs: the extension scratch holds 2
    blobs, so a 6-blob batch (a pass of its own) is extended in three sub-passes, with the same results."""
    batches = [d2.tx([0, 1, 2, 3, 4, 5]), d2.tx([6]), d2.tx([7, 2])]
    bl, com, pr = d2.tx([1, 2, 3, 4, 5, 6])
    batches.append((bl, com, pr[:5 * 128 + 3] + [pr[0]] + pr[5 * 128 + 4:]))      # wrong proof in the last sub-pass
    want = _new(lw, batches, d2.s)
    assert want[0] == [True, True, True, False] and want[1] == [0] * 4
    lw.set_option("cell_chunk_blobs", 2)
    try:
        s = _load(lw, 2)
        try:
            assert _new(lw, batches, s) == want
        finally:
            s.free()
    finally:
        lw.set_option("cell_chunk_blobs", 888)
