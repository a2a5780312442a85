"""GPU tier: commitments, cells and cell proofs in one pass, lwkzg_commit_and_compute_cells_and_kzg_proofs_batch[_device]
(include/lwkzg.h part 3).

Every blob must get exactly the bytes of the two calls the new one replaces: lwkzg_blob_to_kzg_commitment_batch for its
commitment, lwkzg_compute_cells_and_kzg_proofs_batch for its cells and proofs."""
import ctypes
import hashlib
import json
import os

import pytest

from tests.golden.make_cell_fixtures import make_blob

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
R = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
CELL, PROOFS = 128 * 2048, 128 * 48


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


class Mode:
    def __init__(self, lw, mode):
        self.mode, self.s = mode, _load(lw, mode)
        self.order = "little" if mode == 1 else "big"

    def word(self, v):
        return v.to_bytes(32, self.order)

    def bad(self, blob, at=4000):
        """blob with word `at` >= r (a word whose reduction is an ordinary field element)"""
        return blob[:32 * at] + self.word(R + 12345) + blob[32 * at + 32:]


@pytest.fixture(scope="module", params=[2, 0, 1], ids=["mode2", "mode0", "mode1"])
def m(request, lw):
    d = Mode(lw, request.param)
    yield d
    d.s.free()


def _composition(lw, blobs, s):
    """(commitments, cells, proofs, statuses) of the two existing calls; statuses agree between them"""
    n = len(blobs)
    coms, st1 = lw.blob_to_kzg_commitment_batch(b"".join(blobs), n, s)
    cells, proofs, st2 = lw.compute_cells_and_kzg_proofs_batch(b"".join(blobs), n, s)
    assert st1 == st2
    return coms, cells, proofs, st1


def _blobs(m, n, seed):
    return [make_blob(seed + i, m.mode) for i in range(n)]


def _same_as_composition(got, want, skip=()):
    g_c, g_cells, g_p, g_st = got
    w_c, w_cells, w_p, w_st = want
    assert g_st == w_st
    for i in range(len(w_c)):
        if i in skip:
            continue
        assert g_c[i] == w_c[i], i
        assert g_p[i * PROOFS: (i + 1) * PROOFS] == w_p[i * PROOFS: (i + 1) * PROOFS], i
        if g_cells:
            assert g_cells[i * CELL: (i + 1) * CELL] == w_cells[i * CELL: (i + 1) * CELL], i


def test_known_answers(lw, m):
    """The blobs of tests/golden/cell_kats.json: cells and proofs equal the stored answers, commitments the oracle's."""
    kats = [e for e in json.load(open(os.path.join(GOLDEN, "cell_kats.json"))) if e["mode"] == m.mode]
    blobs = [make_blob(e["seed"], m.mode) for e in kats]
    coms, cells, proofs, st = lw.commit_and_compute_cells_and_kzg_proofs_batch(b"".join(blobs), len(blobs), m.s, want_cells=True)
    assert st == [0] * len(blobs)
    for i, e in enumerate(kats):
        assert hashlib.sha256(cells[i * CELL: (i + 1) * CELL]).hexdigest() == e["cells_sha256"]
        assert [proofs[i * PROOFS + 48 * k: i * PROOFS + 48 * k + 48].hex() for k in e["proof_cells"]] == e["proofs"]
        assert coms[i].hex() == e["commitment"]


def test_same_bytes_as_composition(lw, m):
    """8 random blobs, the all-zero blob and a blob of maximal canonical words, with and without cells."""
    blobs = _blobs(m, 8, 800) + [bytes(131072), m.word(R - 1) * 4096]
    want = _composition(lw, blobs, m.s)
    assert want[3] == [0] * 10
    got = lw.commit_and_compute_cells_and_kzg_proofs_batch(b"".join(blobs), 10, m.s, want_cells=True)
    _same_as_composition(got, want)
    coms, cells, proofs, st = lw.commit_and_compute_cells_and_kzg_proofs_batch(b"".join(blobs), 10, m.s)
    assert cells == b"" and (coms, proofs, st) == (got[0], got[2], got[3])


def _raw_host(lw, blobs, s, with_cells=True, with_status=True):
    """the host call on buffers holding sentinel bytes -> (rc, commitments, cells, proofs, status)"""
    n = len(blobs)
    coms = ctypes.create_string_buffer(b"\xab" * (48 * n), 48 * n)
    cells = ctypes.create_string_buffer(b"\xcd" * (CELL * n), CELL * n) if with_cells else None
    proofs = ctypes.create_string_buffer(b"\xef" * (PROOFS * n), PROOFS * n)
    st = (ctypes.c_int * n)(*([-7] * n)) if with_status else None
    rc = lw.load_library().lwkzg_commit_and_compute_cells_and_kzg_proofs_batch(coms, cells, proofs, b"".join(blobs), n, s.ptr, st)
    return rc, coms.raw, cells.raw if with_cells else b"", proofs.raw, list(st) if with_status else None


def _check_failed(res, n, bad, sentinel):
    """the slots of blob `bad` hold `sentinel`; returns the result as (commitments list, cells, proofs, status)"""
    rc, coms, cells, proofs, st = res
    assert coms[48 * bad: 48 * bad + 48] == sentinel[0] * 48
    assert proofs[PROOFS * bad: PROOFS * (bad + 1)] == sentinel[2] * PROOFS
    if cells:
        assert cells[CELL * bad: CELL * (bad + 1)] == sentinel[1] * CELL
    return [coms[48 * i: 48 * i + 48] for i in range(n)], cells, proofs, st


def test_invalid_blob(lw, m):
    """A word >= r in the middle blob: C_KZG_BADARGS and untouched slots for it (modes 1 and 2), every other blob as the
    composition gives it; with status == NULL the call returns that code.  Mode 0 reduces the word: no failure."""
    blobs = _blobs(m, 5, 820)
    blobs[2] = m.bad(blobs[2])
    want = _composition(lw, blobs, m.s)
    if m.mode == 0:
        assert want[3] == [0] * 5
        _same_as_composition(lw.commit_and_compute_cells_and_kzg_proofs_batch(b"".join(blobs), 5, m.s, want_cells=True), want)
        return
    assert want[3] == [0, 0, lw.C_KZG_BADARGS, 0, 0]
    res = _raw_host(lw, blobs, m.s)
    assert res[0] == lw.C_KZG_OK
    _same_as_composition(_check_failed(res, 5, 2, (b"\xab", b"\xcd", b"\xef")), want, skip={2})
    res = _raw_host(lw, blobs, m.s, with_cells=False, with_status=False)
    assert res[0] == lw.C_KZG_BADARGS
    got = _check_failed(res, 5, 2, (b"\xab", b"", b"\xef"))
    _same_as_composition(got[:3] + (want[3],), want, skip={2})


def test_pass_boundaries(lw, m):
    """Passes of 3 blobs over 7 (3 + 3 + 1, the commitments on the XYZZ kernel), the bad blob in the second pass, host and
    device form; then 8 blobs in one pass at the default size (the batched-affine commitment kernel)."""
    blobs = _blobs(m, 8, 840)
    if m.mode:
        blobs[4] = m.bad(blobs[4], 17)
    want = _composition(lw, blobs[:7], m.s)
    lw.set_option("cell_chunk_blobs", 3)
    try:
        got = lw.commit_and_compute_cells_and_kzg_proofs_batch(b"".join(blobs[:7]), 7, m.s, want_cells=True)
        res = _raw_host(lw, blobs[:7], m.s)
        dev = _device(lw, m, blobs[:7])
    finally:
        lw.set_option("cell_chunk_blobs", 888)
    _same_as_composition(got, want, skip={4} if m.mode else ())
    _same_as_host(dev, got, {4} if m.mode else set())
    if m.mode:
        assert got[3][4] == lw.C_KZG_BADARGS
        _same_as_composition(_check_failed(res, 7, 4, (b"\xab", b"\xcd", b"\xef")), want, skip={4})
    want = _composition(lw, blobs, m.s)
    _same_as_composition(lw.commit_and_compute_cells_and_kzg_proofs_batch(b"".join(blobs), 8, m.s, want_cells=True), want, skip={4} if m.mode else ())


def test_round_trip(lw, m):
    """The outputs, as three transactions, pass lwkzg_verify_blob_cell_kzg_proof_batches; swapping the commitments of two
    blobs fails exactly the transactions holding them."""
    blobs = _blobs(m, 8, 860)
    coms, _, proofs, st = lw.commit_and_compute_cells_and_kzg_proofs_batch(b"".join(blobs), 8, m.s)
    assert st == [0] * 8
    prf = [proofs[48 * k: 48 * k + 48] for k in range(8 * 128)]

    def txs(c):
        return [(blobs[a:b], c[a:b], prf[128 * a: 128 * b]) for a, b in ((0, 3), (3, 5), (5, 8))]

    assert lw.verify_blob_cell_kzg_proof_batches(txs(coms), m.s) == ([True] * 3, [0] * 3)
    sw = list(coms)
    sw[1], sw[4] = sw[4], sw[1]
    assert lw.verify_blob_cell_kzg_proof_batches(txs(sw), m.s) == ([False, False, True], [0] * 3)
    sw = list(coms)
    sw[5], sw[7] = sw[7], sw[5]
    assert lw.verify_blob_cell_kzg_proof_batches(txs(sw), m.s) == ([True, True, False], [0] * 3)


def _device(lw, m, blobs, with_status=True, with_cells=True):
    """the device form on torch tensors on a non-default stream, the blobs written on it by a kernel right before the call
    -> (commitments list, cells, proofs, status); unwritten bytes read 0x5a, status -7"""
    import torch

    n = len(blobs)
    src = torch.frombuffer(bytearray(b"".join(blobs)), dtype=torch.uint8).cuda()
    d_c = torch.full((n * 48,), 0x5A, dtype=torch.uint8, device="cuda")
    d_cells = torch.full((n * CELL,), 0x5A, dtype=torch.uint8, device="cuda")
    d_p = torch.full((n * PROOFS,), 0x5A, dtype=torch.uint8, device="cuda")
    d_st = torch.full((n,), -7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        d_b = torch.add(src, 0)
        lw.commit_and_compute_cells_and_kzg_proofs_batch_device(d_c.data_ptr(), d_cells.data_ptr() if with_cells else 0, d_p.data_ptr(), d_b.data_ptr(), n,
                                                                m.s, stream.cuda_stream, d_st.data_ptr() if with_status else 0)
        coms, cells, proofs, st = bytes(d_c.cpu().numpy()), bytes(d_cells.cpu().numpy()), bytes(d_p.cpu().numpy()), d_st.cpu().tolist()
    torch.cuda.synchronize()
    return [coms[48 * i: 48 * i + 48] for i in range(n)], cells, proofs, st


def _same_as_host(got, want, bad, with_status=True, with_cells=True):
    """device-form result against the host form's: failed blobs zeroed, cells 0x5a when not asked for"""
    coms, cells, proofs, st = got
    assert st == (want[3] if with_status else [-7] * len(coms))
    for i in range(len(coms)):
        if i in bad:
            assert coms[i] == bytes(48) and proofs[PROOFS * i: PROOFS * (i + 1)] == bytes(PROOFS)
            assert cells[CELL * i: CELL * (i + 1)] == (bytes(CELL) if with_cells else b"\x5a" * CELL)
            continue
        assert coms[i] == want[0][i], i
        assert proofs[PROOFS * i: PROOFS * (i + 1)] == want[2][PROOFS * i: PROOFS * (i + 1)], i
        assert cells[CELL * i: CELL * (i + 1)] == (want[1][CELL * i: CELL * (i + 1)] if with_cells else b"\x5a" * CELL), i


def test_device_form(lw, m):
    """Torch tensors on a non-default stream, the blobs written on it right before the call: with and without d_status
    and d_cells, the host form's bytes, failed blobs zeroed."""
    blobs = _blobs(m, 6, 880)
    if m.mode:
        blobs[3] = m.bad(blobs[3], 0)
    want = lw.commit_and_compute_cells_and_kzg_proofs_batch(b"".join(blobs), 6, m.s, want_cells=True)
    bad = {3} if m.mode else set()
    assert want[3] == [lw.C_KZG_BADARGS if i in bad else 0 for i in range(6)]
    for with_status in (True, False):
        for with_cells in (True, False):
            _same_as_host(_device(lw, m, blobs, with_status, with_cells), want, bad, with_status, with_cells)


def test_whole_call_errors(lw, m):
    """n == 0 writes nothing; a NULL blobs, commitments or proofs is C_KZG_BADARGS, host and device form alike;
    settings without the monomial SRS are C_KZG_ERROR."""
    from lambdaworks_kzg_b200.api import CKZGSettings

    lib = lw.load_library()
    f, g = lib.lwkzg_commit_and_compute_cells_and_kzg_proofs_batch, lib.lwkzg_commit_and_compute_cells_and_kzg_proofs_batch_device
    blobs = b"".join(_blobs(m, 2, 900))
    coms = ctypes.create_string_buffer(b"\xab" * 96, 96)
    cells = ctypes.create_string_buffer(b"\xcd" * (2 * CELL), 2 * CELL)
    proofs = ctypes.create_string_buffer(b"\xef" * (2 * PROOFS), 2 * PROOFS)
    st = (ctypes.c_int * 2)(-7, -7)
    assert f(coms, cells, proofs, blobs, 0, m.s.ptr, st) == lw.C_KZG_OK
    assert f(None, None, None, None, 0, m.s.ptr, None) == lw.C_KZG_OK
    for k in range(3):
        args = [coms, proofs, blobs]
        args[k] = None
        assert f(args[0], cells, args[1], args[2], 2, m.s.ptr, st) == lw.C_KZG_BADARGS
    assert coms.raw == b"\xab" * 96 and cells.raw == b"\xcd" * (2 * CELL) and proofs.raw == b"\xef" * (2 * PROOFS) and list(st) == [-7, -7]
    assert g(1 << 20, 1 << 20, 1 << 20, 1 << 20, 0, m.s.ptr, None, 1 << 20) == lw.C_KZG_OK
    assert g(None, None, None, None, 0, m.s.ptr, None, None) == lw.C_KZG_OK
    for k in range(3):
        args = [1 << 20, 1 << 20, 1 << 20]
        args[k] = None
        assert g(args[0], 1 << 20, args[1], args[2], 2, m.s.ptr, None, None) == lw.C_KZG_BADARGS
    if m.mode == 0:
        return
    # hand-built Lagrange settings carry no monomial SRS
    g1 = ctypes.create_string_buffer(m.s.g1_values_bytes(), 4096 * 144)
    g2 = ctypes.create_string_buffer(m.s.g2_values_bytes(), 65 * 288)
    lw.set_option("mode", m.mode)
    lw.set_option("window_bits", 8)
    try:
        s = CKZGSettings(None, ctypes.cast(g1, ctypes.c_void_p), ctypes.cast(g2, ctypes.c_void_p))
        with pytest.raises(lw.KzgError) as e:
            lw.commit_and_compute_cells_and_kzg_proofs_batch(blobs, 2, s)
        assert e.value.code == lw.C_KZG_ERROR
    finally:
        lw.set_option("mode", 0)
        lw.set_option("window_bits", 13)


def test_two_gpus(lw, m):
    """After set_devices([0, 1]) the host form shards the blobs over both GPUs, with the same bytes."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    blobs = _blobs(m, 8, 920)
    if m.mode:
        blobs[5] = m.bad(blobs[5])
    want = lw.commit_and_compute_cells_and_kzg_proofs_batch(b"".join(blobs), 8, m.s, want_cells=True)
    lw.set_devices([0, 1])
    try:
        got = lw.commit_and_compute_cells_and_kzg_proofs_batch(b"".join(blobs), 8, m.s, want_cells=True)
    finally:
        lw.set_devices([])
    assert got == want
