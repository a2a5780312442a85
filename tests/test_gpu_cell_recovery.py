"""GPU tier: batched cell recovery, lwkzg_recover_cells_and_kzg_proofs_batch[_device] (include/lwkzg.h part 3).

Good blobs must give the bytes of compute_cells_and_kzg_proofs on the original blobs (and of the single
recover_cells_and_kzg_proofs call); a failed blob gets its own status without touching the others."""
import ctypes
import hashlib
import json
import os
import random

import pytest

from tests.golden.make_cell_fixtures import make_blob

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
R = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
CB = 128 * 2048     # cells of one blob
PB = 128 * 48       # proofs of one blob
SENTINEL = 0xA5


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


@pytest.fixture(scope="module")
def s2(lw):
    s = _load(lw, 2)
    yield s
    s.free()


@pytest.fixture(scope="module")
def ref230(lw, s2):
    """230 synthetic blobs with all their cells and proofs from the compute batch."""
    n = 230
    blobs = b"".join(lw.synth_blob_host(k) for k in range(n))
    cells, proofs, st = lw.compute_cells_and_kzg_proofs_batch(blobs, n, s2)
    assert st == [0] * n
    return cells, proofs


def _cell(cells, b, i):
    return cells[(b * 128 + i) * 2048: (b * 128 + i + 1) * 2048]


def _select(cells, blobs_and_indices):
    """(blob index into `cells`, index list) per output blob -> flat indices, flat cell bytes"""
    idx, sel = [], []
    for b, keep in blobs_and_indices:
        idx += keep
        sel += [_cell(cells, b, i) for i in keep]
    return idx, b"".join(sel)


def _raw_batch(lw, idx, cells, num_cells, n, s, status=True, fill=SENTINEL):
    """the C call on sentinel-filled host buffers -> (return code, cells, proofs, status or None)"""
    rc = ctypes.create_string_buffer(bytes([fill]) * max(1, n * CB))
    rp = ctypes.create_string_buffer(bytes([fill]) * max(1, n * PB))
    st = (ctypes.c_int * max(1, n))(*([-7] * max(1, n))) if status else None
    ix = (ctypes.c_uint64 * max(1, len(idx)))(*idx)
    code = lw.load_library().lwkzg_recover_cells_and_kzg_proofs_batch(rc, rp, ix, cells or b"\0", num_cells, n, s.ptr, st)
    return code, rc.raw[: n * CB], rp.raw[: n * PB], (list(st)[:n] if status else None)


def _device_batch(lw, torch, idx, cells, num_cells, n, s, fill=SENTINEL):
    d_idx = torch.tensor(idx, dtype=torch.int64, device="cuda")
    d_in = torch.frombuffer(bytearray(cells), dtype=torch.uint8).cuda()
    d_c = torch.full((n * CB,), fill, dtype=torch.uint8, device="cuda")
    d_p = torch.full((n * PB,), fill, dtype=torch.uint8, device="cuda")
    d_st = torch.full((n,), -7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    lw.recover_cells_and_kzg_proofs_batch_device(d_c.data_ptr(), d_p.data_ptr(), d_idx.data_ptr(), d_in.data_ptr(), num_cells, n, s,
                                                 torch.cuda.current_stream().cuda_stream, d_st.data_ptr())
    torch.cuda.synchronize()
    return bytes(d_c.cpu().numpy()), bytes(d_p.cpu().numpy()), d_st.tolist()


def test_batch_equals_single_calls(lw, s2):
    """Six blobs with six different 64-cell index sets in one call, one blob from 101 cells in another; cells only
    and proofs only as well."""
    rng = random.Random(5)
    blobs = [make_blob(60 + i, 2) for i in range(6)]
    singles = [lw.compute_cells_and_kzg_proofs(b, s2) for b in blobs]
    full = b"".join(b"".join(cs) for cs, _ in singles)
    want_c = full
    want_p = b"".join(b"".join(ps) for _, ps in singles)
    sets = [sorted(rng.sample(range(128), 64)), list(range(64, 128)), list(range(0, 128, 2)), list(range(1, 128, 2)), list(range(64)),
            sorted(rng.sample(range(128), 64))]
    idx, sel = _select(full, list(enumerate(sets)))
    cells, proofs, st = lw.recover_cells_and_kzg_proofs_batch(idx, sel, 64, 6, s2)
    assert st == [0] * 6
    assert cells == want_c and proofs == want_p
    c_only, none, st = lw.recover_cells_and_kzg_proofs_batch(idx, sel, 64, 6, s2, want_proofs=False)
    assert st == [0] * 6 and c_only == want_c and none == b""
    none, p_only, st = lw.recover_cells_and_kzg_proofs_batch(idx, sel, 64, 6, s2, want_cells=False)
    assert st == [0] * 6 and p_only == want_p and none == b""
    # one blob from 101 cells, against the single recovery call too
    keep = sorted(rng.sample(range(128), 101))
    idx, sel = _select(full, [(2, keep)])
    cells, proofs, st = lw.recover_cells_and_kzg_proofs_batch(idx, sel, 101, 1, s2)
    rc, rp = lw.recover_cells_and_kzg_proofs(keep, [_cell(full, 2, i) for i in keep], s2)
    assert st == [0] and cells == want_c[2 * CB: 3 * CB] == b"".join(rc) and proofs == want_p[2 * PB: 3 * PB] == b"".join(rp)


def test_peerdas_block_host_and_device(lw, s2, ref230):
    """128 blobs sharing one set of 64 columns, through the host and the device API."""
    import torch

    cells, proofs = ref230
    n = 128
    keep = sorted(random.Random(128).sample(range(128), 64))
    idx, sel = _select(cells, [(b, keep) for b in range(n)])
    rc, rp, st = lw.recover_cells_and_kzg_proofs_batch(idx, sel, 64, n, s2)
    assert st == [0] * n
    assert rc == cells[: n * CB] and rp == proofs[: n * PB]
    dc, dp, dst = _device_batch(lw, torch, idx, sel, 64, n, s2)
    assert dst == [0] * n and dc == rc and dp == rp


def test_batched_affine_threshold_and_pass_offsets(lw, s2, ref230):
    """230 blobs: the FK20 pass crosses CELL_BA_MIN_BLOBS (224); 5 blobs in passes of 2 + 2 + 1."""
    cells, proofs = ref230
    rng = random.Random(230)
    sets = [sorted(rng.sample(range(128), 64)) for _ in range(230)]
    idx, sel = _select(cells, list(enumerate(sets)))
    rc, rp, st = lw.recover_cells_and_kzg_proofs_batch(idx, sel, 64, 230, s2)
    assert st == [0] * 230 and rc == cells and rp == proofs
    pick = [3, 99, 150, 7, 229]
    idx, sel = _select(cells, [(b, sets[b]) for b in pick])
    lw.set_option("cell_chunk_blobs", 2)
    try:
        rc, rp, st = lw.recover_cells_and_kzg_proofs_batch(idx, sel, 64, 5, s2)
    finally:
        lw.set_option("cell_chunk_blobs", 888)
    assert st == [0] * 5
    for k, b in enumerate(pick):
        assert rc[k * CB: (k + 1) * CB] == cells[b * CB: (b + 1) * CB]
        assert rp[k * PB: (k + 1) * PB] == proofs[b * PB: (b + 1) * PB]


def _failure_batch(full):
    """eight blobs of 66 cells from `full` (the cells of blobs 0..7): good ones around five malformed ones.  66, not 64:
    any 64 cells fit a polynomial of degree < 4096, so only more of them can be inconsistent."""
    base = sorted(list(range(0, 128, 2)) + [1, 3])
    plan = []
    for b in range(8):
        keep = list(base)
        cells = [_cell(full, b, i) for i in keep]
        if b == 1:     # unsorted
            keep[3], keep[4] = keep[4], keep[3]
            cells[3], cells[4] = cells[4], cells[3]
        elif b == 3:   # repeated
            keep[5] = keep[4]
            cells[5] = cells[4]
        elif b == 4:   # index 128
            keep[-1] = 128
        elif b == 5:   # a word >= r
            cells[10] = cells[10][:64] + R.to_bytes(32, "big") + cells[10][96:]
        elif b == 6:   # inconsistent: cell 3's values under index 1
            cells[1] = cells[3]
        plan.append((keep, cells))
    return [i for keep, _ in plan for i in keep], b"".join(c for _, cells in plan for c in cells), [1, 3, 4, 5, 6]


@pytest.mark.parametrize("mode", [2, 0])
def test_per_blob_failures_inside_a_batch(lw, s2, mode):
    import torch

    s = s2 if mode == 2 else _load(lw, 0)
    try:
        blobs = [make_blob(80 + b, mode) for b in range(8)]
        full, proofs, st = lw.compute_cells_and_kzg_proofs_batch(b"".join(blobs), 8, s)
        assert st == [0] * 8
        idx, sel, bad = _failure_batch(full)
        code = lw.C_KZG_BADARGS if mode == 2 else lw.C_KZG_ERROR
        want_st = [code if b in bad else 0 for b in range(8)]
        rc_code, hc, hp, hst = _raw_batch(lw, idx, sel, 66, 8, s)
        assert rc_code == lw.C_KZG_OK and hst == want_st
        for b in range(8):
            if b in bad:
                assert hc[b * CB: (b + 1) * CB] == bytes([SENTINEL]) * CB and hp[b * PB: (b + 1) * PB] == bytes([SENTINEL]) * PB, b
            else:
                assert hc[b * CB: (b + 1) * CB] == full[b * CB: (b + 1) * CB] and hp[b * PB: (b + 1) * PB] == proofs[b * PB: (b + 1) * PB], b
        dc, dp, dst = _device_batch(lw, torch, idx, sel, 66, 8, s)
        assert dst == hst
        for b in range(8):
            if b in bad:
                assert dc[b * CB: (b + 1) * CB] == bytes(CB) and dp[b * PB: (b + 1) * PB] == bytes(PB), b
            else:
                assert dc[b * CB: (b + 1) * CB] == hc[b * CB: (b + 1) * CB] and dp[b * PB: (b + 1) * PB] == hp[b * PB: (b + 1) * PB], b
        # status == NULL: the first failing blob's code
        rc_code, _, _, _ = _raw_batch(lw, idx, sel, 66, 8, s, status=False)
        assert rc_code == code
        # the single call agrees with the batch on every blob
        for b in range(8):
            k = idx[b * 66: (b + 1) * 66]
            cs = [sel[(b * 66 + j) * 2048: (b * 66 + j + 1) * 2048] for j in range(66)]
            if b in bad:
                with pytest.raises(lw.KzgError) as ei:
                    lw.recover_cells_and_kzg_proofs(k, cs, s)
                assert ei.value.code == code, b
            else:
                rc, rp = lw.recover_cells_and_kzg_proofs(k, cs, s)
                assert b"".join(rc) == hc[b * CB: (b + 1) * CB] and b"".join(rp) == hp[b * PB: (b + 1) * PB]
    finally:
        if s is not s2:
            s.free()


def test_whole_call_errors(lw, s2):
    import torch

    cells, _, _ = lw.compute_cells_and_kzg_proofs_batch(make_blob(90, 2), 1, s2)
    for num_cells in (63, 129):
        keep = list(range(num_cells)) if num_cells <= 128 else list(range(128)) + [0]
        idx, sel = keep, b"".join(_cell(cells, 0, i % 128) for i in keep)
        code, hc, _, st = _raw_batch(lw, idx, sel, num_cells, 1, s2)
        assert code == lw.C_KZG_BADARGS and hc == bytes([SENTINEL]) * CB and st == [-7]
        with pytest.raises(lw.KzgError) as ei:
            lw.recover_cells_and_kzg_proofs_batch_device(1 << 20, 1 << 20, 1 << 20, 1 << 20, num_cells, 1, s2)
        assert ei.value.code == lw.C_KZG_BADARGS
    lib = lw.load_library()
    keep = list(range(64))
    ix = (ctypes.c_uint64 * 64)(*keep)
    sel = b"".join(_cell(cells, 0, i) for i in keep)
    out_c = ctypes.create_string_buffer(CB)
    out_p = ctypes.create_string_buffer(PB)
    st = (ctypes.c_int * 1)()
    assert lib.lwkzg_recover_cells_and_kzg_proofs_batch(out_c, out_p, None, sel, 64, 1, s2.ptr, st) == lw.C_KZG_BADARGS
    assert lib.lwkzg_recover_cells_and_kzg_proofs_batch(out_c, out_p, ix, None, 64, 1, s2.ptr, st) == lw.C_KZG_BADARGS
    assert lib.lwkzg_recover_cells_and_kzg_proofs_batch(None, None, ix, sel, 64, 1, s2.ptr, st) == lw.C_KZG_BADARGS
    for args in ((1 << 20, 1 << 20, None, 1 << 20), (1 << 20, 1 << 20, 1 << 20, None), (None, None, 1 << 20, 1 << 20)):
        assert lib.lwkzg_recover_cells_and_kzg_proofs_batch_device(*args, 64, 1, s2.ptr, None, None) == lw.C_KZG_BADARGS
    # n == 0: OK and nothing written
    st0 = (ctypes.c_int * 1)(-7)
    fill = ctypes.create_string_buffer(bytes([SENTINEL]) * CB)
    assert lib.lwkzg_recover_cells_and_kzg_proofs_batch(fill, None, ix, sel, 64, 0, s2.ptr, st0) == lw.C_KZG_OK
    assert fill.raw[:CB] == bytes([SENTINEL]) * CB and st0[0] == -7
    d_c = torch.full((CB,), SENTINEL, dtype=torch.uint8, device="cuda")
    lw.recover_cells_and_kzg_proofs_batch_device(d_c.data_ptr(), 0, 1 << 20, 1 << 20, 64, 0, s2)
    torch.cuda.synchronize()
    assert bool((d_c == SENTINEL).all())


@pytest.mark.parametrize("mode", [0, 1])
def test_reference_and_le_modes(lw, py_setup, mode):
    """The batch in modes 0 and 1 against the committed cell known answers and the oracle's recovery."""
    from oracle.py import cells as ocells

    o = ocells.CellOracle(py_setup, mode)
    kat = [e for e in json.load(open(os.path.join(GOLDEN, "cell_kats.json"))) if e["mode"] == mode][0]
    s = _load(lw, mode)
    try:
        blobs = [make_blob(kat["seed"], mode), make_blob(kat["seed"] + 100, mode), make_blob(kat["seed"] + 200, mode)]
        full, proofs, st = lw.compute_cells_and_kzg_proofs_batch(b"".join(blobs), 3, s)
        assert st == [0] * 3
        sets = [list(range(1, 128, 2)), list(range(64, 128)), sorted(random.Random(mode).sample(range(128), 64))]
        idx, sel = _select(full, list(enumerate(sets)))
        rc, rp, st = lw.recover_cells_and_kzg_proofs_batch(idx, sel, 64, 3, s)
        assert st == [0] * 3 and rc == full and rp == proofs
        assert hashlib.sha256(rc[:CB]).hexdigest() == kat["cells_sha256"]
        assert [rp[48 * i: 48 * i + 48].hex() for i in kat["proof_cells"]] == kat["proofs"]
        # the oracle's own recovery of blob 2 from its index set
        want_c, want_p = o.recover_cells_and_kzg_proofs(sets[2], [_cell(full, 2, i) for i in sets[2]], cell_subset=[0, 77])
        assert rc[2 * CB: 3 * CB] == b"".join(want_c)
        assert [rp[(2 * 128 + i) * 48: (2 * 128 + i + 1) * 48] for i in (0, 77)] == want_p
    finally:
        s.free()


def test_stream_ordering(lw, s2, ref230):
    """The input cells arrive by a copy enqueued on a non-default torch stream right before the call, and the outputs
    are read on that stream without a device synchronize."""
    import torch

    cells, proofs = ref230
    n = 128
    keep = list(range(64, 128))
    idx, sel = _select(cells, [(b, keep) for b in range(n)])
    host = torch.frombuffer(bytearray(sel), dtype=torch.uint8).pin_memory()
    d_in = torch.zeros(len(sel), dtype=torch.uint8, device="cuda")
    d_idx = torch.tensor(idx, dtype=torch.int64, device="cuda")
    d_c = torch.zeros(n * CB, dtype=torch.uint8, device="cuda")
    d_p = torch.zeros(n * PB, dtype=torch.uint8, device="cuda")
    d_st = torch.full((n,), -7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        d_in.copy_(host, non_blocking=True)
        lw.recover_cells_and_kzg_proofs_batch_device(d_c.data_ptr(), d_p.data_ptr(), d_idx.data_ptr(), d_in.data_ptr(), 64, n, s2,
                                                     side.cuda_stream, d_st.data_ptr())
        out_c, out_p, out_st = d_c.cpu(), d_p.cpu(), d_st.cpu()
    assert out_st.tolist() == [0] * n
    assert bytes(out_c.numpy()) == cells[: n * CB] and bytes(out_p.numpy()) == proofs[: n * PB]
