"""CPU tier: the forgery helpers of tests/_forge.py, checked against the oracle in every mode.  A forged pair must be
rejected by the oracle's batch verification and accepted by the batch equation under equal weights -- otherwise
the GPU soundness tests built on it would prove nothing."""
import dataclasses
import random

import pytest

from oracle.py import bls, cells, kzg
from tests import _forge

R = bls.R
MODES = [0, 1, 2]
MODE_IDS = ["ref", "ckzg_le", "deneb"]


@pytest.fixture(scope="module", params=MODES, ids=MODE_IDS)
def batch(request, py_setup):
    """(mode, oracle, 5 valid items)."""
    mode = request.param
    o = _forge.oracle_for(mode, py_setup)
    rnd = random.Random(4844 + mode)
    items = [_forge.make_item(o, _forge.random_blob(mode, rnd)) for _ in range(5)]
    return mode, o, items


def _cols(items):
    return [t.blob for t in items], [t.commitment for t in items], [t.proof for t in items]


def test_items_are_valid_and_their_logs_match_the_points(batch):
    mode, o, items = batch
    for t in items:
        assert t.commitment == o.blob_to_kzg_commitment(t.blob)
        assert t.proof == o.compute_blob_kzg_proof(t.blob, t.commitment)
        assert t.commitment == bls.g1_compress(bls.g1_mul(bls.G1, t.c_log))
        assert t.proof == bls.g1_compress(bls.g1_mul(bls.G1, t.pi_log))
    assert o.verify_blob_kzg_proof_batch(*_cols(items)) is True


@pytest.mark.parametrize("n,pair", [(3, (0, 2)), (5, (0, 1)), (5, (1, 4))])
def test_forged_pair_passes_equal_weights_only(batch, n, pair):
    mode, o, items = batch
    blobs, coms, proofs = _cols(items[:n])
    i, j = pair
    forged = _forge.forge_blob_batch(o, blobs, coms, proofs, i, j)
    assert [k for k in range(n) if forged[k] != proofs[k]] == [i, j]
    assert o.verify_blob_kzg_proof_batch(blobs, coms, forged) is False
    assert _forge.weighted_batch_check(o, blobs, coms, forged, [1] * n) is True
    assert _forge.weighted_batch_check(o, blobs, coms, forged, [12345] * n) is True
    # weights equal only on the pair still pass; any difference on the pair fails
    w = [3, 5, 7, 11, 13][:n]
    w[j] = w[i]
    assert _forge.weighted_batch_check(o, blobs, coms, forged, w) is True
    w[j] = w[i] + 1
    assert _forge.weighted_batch_check(o, blobs, coms, forged, w) is False
    # the batch challenge weights r^i are the oracle's verdict, for the valid batch and the forged one
    zs = [_forge.challenge(o, b, c) for b, c in zip(blobs, coms)]
    ys = [_forge.poly_at(o, b, z) for b, z in zip(blobs, zs)]
    r = _forge.batch_challenge(mode, coms, zs, ys, forged)
    assert _forge.weighted_batch_check(o, blobs, coms, forged, [pow(r, k, R) for k in range(n)]) is False
    r = _forge.batch_challenge(mode, coms, zs, ys, proofs)
    assert _forge.weighted_batch_check(o, blobs, coms, proofs, [pow(r, k, R) for k in range(n)]) is True


def test_batch_challenge_matches_the_oracle(batch):
    mode, o, items = batch
    if mode == 1:
        pytest.skip("the MODE_CKZG_LE oracle verifies a batch item by item: it has no batch challenge")
    coms = [t.commitment for t in items]
    proofs = [t.proof for t in items]
    zs, ys = [t.z for t in items], [t.y for t in items]
    if mode == 0:
        want = o.batch_challenge([bls.g1_decompress(c) for c in coms], zs, ys, [bls.g1_decompress(p) for p in proofs])
    else:
        want = o.batch_challenge(coms, zs, ys, proofs)
    assert _forge.items_challenge(mode, items) == want


def test_non_g1_points_are_rejected_with_the_mode_code(batch):
    mode, o, items = batch
    code = _forge.decode_error_code(mode)
    pts = _forge.non_g1_points()
    assert len(set(pts)) == 2
    for enc in pts:
        x =int.from_bytes(bytes([enc[0] & 0x1F]) + enc[1:], "big")
        y = bls.fp_sqrt(x ** 3 + 4)
        assert y is not None, "not on the curve"
        assert not bls.g1_in_subgroup((x, y)) and not bls.g1_in_subgroup((x, bls.P - y))
        with pytest.raises(kzg.KzgError) as e:
            o._decompress(enc)
        assert e.value.code == code
        blobs, coms, proofs = _cols(items[:3])
        for role in ("commitment", "proof"):
            c2, p2 = list(coms), list(proofs)
            (c2 if role == "commitment" else p2)[1] = enc
            with pytest.raises(kzg.KzgError) as e:
                o.verify_blob_kzg_proof_batch(blobs, c2, p2)
            assert e.value.code == code, role


def test_expected_partial(batch):
    mode, o, items = batch
    r = _forge.items_challenge(mode, items)
    whole = _forge.expected_partial(items, r, 0)
    assert len(whole) == 288 and whole[96:192] == bytes(96)
    assert _forge.phase3(whole, o.s.tau) is True
    # the same sums from the points themselves
    w = [pow(r, k, R) for k in range(len(items))]
    pis = [bls.g1_decompress(t.proof) for t in items]
    s1 = bls.g1_sum(bls.g1_mul(p, wk) for p, wk in zip(pis, w))
    s3 = bls.g1_sum([bls.g1_mul(p, wk * t.z % R) for p, wk, t in zip(pis, w, items)] +
                    [bls.g1_mul(bls.g1_decompress(t.commitment), wk) for wk, t in zip(w, items)] +
                    [bls.g1_neg(bls.g1_mul(bls.G1, sum(wk * t.y for wk, t in zip(w, items)) % R))])
    assert whole == _forge._be96(s1) + bytes(96) + _forge._be96(s3)
    # split over ranks: the per-rank partials pass together, and only with the right offsets
    parts = _forge.expected_partial(items[:2], r, 0) + _forge.expected_partial(items[2:], r, 2)
    assert _forge.phase3(parts, o.s.tau) is True
    assert _forge.expected_partial([], r, 0) == bytes(288)
    # a forged pair: its partial fails phase 3 under r^i and passes when both items get the same weight
    b = (-_forge.DEFAULT_A * (o.s.tau - items[0].z) * bls.fr_inv((o.s.tau - items[3].z) % R)) % R
    forged = list(items)
    forged[0] = dataclasses.replace(items[0], pi_log=(items[0].pi_log + _forge.DEFAULT_A) % R)
    forged[3] = dataclasses.replace(items[3], pi_log=(items[3].pi_log + b) % R)
    assert _forge.phase3(_forge.expected_partial(forged, r, 0), o.s.tau) is False
    same = _forge.expected_partial(forged[:3], r, 0) + _forge.expected_partial(forged[3:], r, 0)   # item 3 weighted r^0
    assert _forge.phase3(same, o.s.tau) is True


@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_forged_cell_pairs(py_setup, mode):
    co = cells.CellOracle(py_setup, mode)
    o = _forge.oracle_for(mode, py_setup)
    rnd = random.Random(77 + mode)
    blobs = [_forge.random_blob(mode, rnd) for _ in range(2)]
    want = {0: [3, 9, 70], 1: [9, 120]}
    cl, pl = {}, {}
    for b, idx in want.items():
        cs, ps = co.compute_cells_and_kzg_proofs(blobs[b], cell_subset=idx)
        for k, p in zip(idx, ps):
            cl[b, k], pl[b, k] = cs[k], p
    coms = [o.blob_to_kzg_commitment(b) for b in blobs]
    tau = py_setup.tau
    batches = {
        "two cells of one blob": ([(0, 3), (0, 9), (0, 70)], 0, 2),
        "one cell index, two blobs": ([(0, 3), (0, 9), (1, 120), (1, 9)], 1, 3),
    }
    for name, (sel, i, j) in batches.items():
        c = [coms[b] for b, _ in sel]
        idx = [k for _, k in sel]
        cel = [cl[s] for s in sel]
        prf = [pl[s] for s in sel]
        assert co.verify_cell_kzg_proof_batch(c, idx, cel, prf) is True, name
        assert _forge.weighted_cell_check(co, c, idx, cel, prf, [5, 6, 7, 8][:len(sel)]) is True, name
        forged = _forge.forge_cell_batch(tau, idx, prf, i, j)
        assert co.verify_cell_kzg_proof_batch(c, idx, cel, forged) is False, name
        assert _forge.weighted_cell_check(co, c, idx, cel, forged, [1] * len(sel)) is True, name
        w = [5, 6, 7, 8][:len(sel)]
        assert _forge.weighted_cell_check(co, c, idx, cel, forged, w) is False, name
    # a proof outside G1 is rejected with the mode's code
    for enc in _forge.non_g1_points():
        with pytest.raises(kzg.KzgError) as e:
            co.verify_cell_kzg_proof_batch([coms[0]], [3], [cl[0, 3]], [enc])
        assert e.value.code == co.bad
