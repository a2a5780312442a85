"""GPU tier: batched verification is sound only because item i of a batch is weighted by r^(first + i).  A valid batch
verifies under any weights, and one bad proof (or a swapped pair) fails under any weights, so the other tests cannot
tell correct weights from wrong ones.  These can:

* phase 1 / phase 2 output bytes against the oracle (tests/_forge.py expected_partial, from discrete logs), for
  uneven shards over 1, 2 and 3 simulated ranks;
* forged proof pairs that pass exactly when their two weights are equal, placed where a weight bug would make them
  equal (neighbours, one RLC block apart, one chunk / staging super-batch apart, the same local index on two ranks),
  through every entry point, in all three modes;
* points on the curve but outside G1 on every r-torsion path (decompression, the separate subgroup kernels,
  the deferred check of single verification), followed by a valid batch: no stale status;
* forged cell-proof pairs for verify_cell_kzg_proof_batch."""
import contextlib
import os
from dataclasses import dataclass
from typing import List

import pytest

from oracle.py import cells, kzg
from tests import _forge

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
B = kzg.BYTES_PER_BLOB
N = 300
MODE_IDS = ["ref", "ckzg_le", "deneb"]


@pytest.fixture(scope="module")
def lw():
    import lambdaworks_kzg_b200 as m

    m.load_library()
    return m


@contextlib.contextmanager
def options(lw, **kv):
    old = {k: lw.get_option(k) for k in kv}
    try:
        for k, v in kv.items():
            lw.set_option(k, v)
        yield
    finally:
        for k, v in old.items():
            lw.set_option(k, v)


@dataclass
class Env:
    mode: int
    s: object
    o: object
    items: List[_forge.Item]


@pytest.fixture(scope="module", params=[0, 1, 2], ids=MODE_IDS)
def env(request, lw, py_setup):
    """Settings of one mode with 8-bit windows, and N valid items built by the oracle."""
    import random

    mode = request.param
    with options(lw, mode=mode, window_bits=8, cell_window_bits=8):
        s = lw.load_trusted_setup_file(os.path.join(GOLDEN, "trusted_setup.txt"))
    o = _forge.oracle_for(mode, py_setup)
    rnd = random.Random(7594 + mode)
    items = [_forge.make_item(o, _forge.random_blob(mode, rnd)) for _ in range(N)]
    yield Env(mode, s, o, items)
    s.free()


# ------------------------------------------------------------------ entry points
class Batch:
    """Blobs of one batch, with their device / pinned copies made once."""

    def __init__(self, blobs):
        self.blobs = list(blobs)
        self.n = len(self.blobs)
        self.flat = b"".join(self.blobs)
        self._dev = self._pin = None

    def dev(self):
        if self._dev is None:
            self._dev = _to_dev(self.flat)
        return self._dev

    def pinned(self):
        if self._pin is None:
            self._pin = _to_pinned(self.flat)
        return self._pin


def _to_dev(data: bytes):
    import torch

    t = torch.frombuffer(bytearray(data), dtype=torch.uint8).to("cuda") if data else torch.zeros(1, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()   # the library's streams do not order after torch's
    return t


def _to_pinned(data: bytes):
    import torch

    t = torch.empty(max(len(data), 1), dtype=torch.uint8, pin_memory=True)
    if data:
        t[: len(data)].copy_(torch.frombuffer(bytearray(data), dtype=torch.uint8))
    return t


def v_host(lw, s, bt, coms, proofs):
    return lw.verify_blob_kzg_proof_batch(bt.blobs, coms, proofs, s)


def v_pinned(lw, s, bt, coms, proofs):
    c, p = _to_pinned(b"".join(coms)), _to_pinned(b"".join(proofs))
    return lw.verify_blob_kzg_proof_batch_ptr(bt.pinned().data_ptr(), c.data_ptr(), p.data_ptr(), bt.n, s)


def v_device(lw, s, bt, coms, proofs):
    c, p = _to_dev(b"".join(coms)), _to_dev(b"".join(proofs))
    return lw.verify_blob_kzg_proof_batch_device(bt.dev().data_ptr(), c.data_ptr(), p.data_ptr(), bt.n, s)


def run_phases(lw, s, bt, coms, proofs, world, device):
    """Phases 1 - 3 over `world` simulated ranks on one GPU -> (result, all tuples, partials, r after each phase 2).
    One process: the phase 1 of a rank must directly precede its phase 2, so the tuples are gathered first."""
    n = bt.n
    shards = [lw.shard_range(n, world, r) for r in range(world)]
    rs = []
    if not device:
        def p1(first, cnt):
            return lw.verify_batch_phase1(bt.flat[first * B:(first + cnt) * B], b"".join(coms[first:first + cnt]),
                                          b"".join(proofs[first:first + cnt]), cnt, s)
        all_t = b"".join(p1(f, c) for f, c in shards)
        parts = b""
        for f, c in shards:
            p1(f, c)
            parts += lw.verify_batch_phase2(all_t, n, f, c, s)
            rs.append(lw.debug_batch_challenge(s))
        return lw.verify_batch_phase3(parts, world, s), all_t, parts, rs
    import torch

    d_b, d_c, d_p = bt.dev(), _to_dev(b"".join(coms)), _to_dev(b"".join(proofs))
    d_t = torch.zeros(max(n, 1) * 160, dtype=torch.uint8, device="cuda")
    d_parts = torch.zeros(world * 288, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()

    def p1(first, cnt):
        lw.verify_batch_phase1_device(d_t.data_ptr() + 160 * first, d_b.data_ptr() + B * first, d_c.data_ptr() + 48 * first,
                                      d_p.data_ptr() + 48 * first, cnt, s, True)
    for f, c in shards:
        p1(f, c)
    for rank, (f, c) in enumerate(shards):
        p1(f, c)
        lw.verify_batch_phase2_device(d_parts.data_ptr() + 288 * rank, d_t.data_ptr(), n, f, c, s)
        rs.append(lw.debug_batch_challenge(s))
    ok = lw.verify_batch_phase3_device(d_parts.data_ptr(), world, s)
    return ok, bytes(d_t[: 160 * n].cpu().numpy().tobytes()), bytes(d_parts.cpu().numpy().tobytes()), rs


def entry_points(world=1):
    """name -> f(lw, s, batch, commitments, proofs) -> bool"""
    return {
        "host": v_host,
        "pinned": v_pinned,
        "device": v_device,
        "phases": lambda lw, s, bt, c, p: run_phases(lw, s, bt, c, p, world, False)[0],
        "phases_device": lambda lw, s, bt, c, p: run_phases(lw, s, bt, c, p, world, True)[0],
    }


def cols(items):
    return [t.blob for t in items], [t.commitment for t in items], [t.proof for t in items]


# ------------------------------------------------------------------ a. phase-2 bytes
@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
@pytest.mark.parametrize("n", [1, 2, 127, 128, 129, 300])
def test_phase2_bytes_match_the_oracle(lw, env, n, device):
    items = env.items[:n]
    blobs, coms, proofs = cols(items)
    bt = Batch(blobs)
    r = _forge.items_challenge(env.mode, items)
    want_tuples = _forge.items_tuples(env.mode, items)
    configs = [{}] + ([{"chunk_blobs": 50, "verify_super_blobs": 128}] if n == 300 else [])
    for cfg in configs:
        with options(lw, **cfg):
            for world in (1, 2, 3):
                ok, tuples, parts, rs = run_phases(lw, env.s, bt, coms, proofs, world, device)
                assert tuples == want_tuples, (cfg, world)
                assert rs == [r] * world, (cfg, world)
                for rank in range(world):
                    first, cnt = lw.shard_range(n, world, rank)
                    want = _forge.expected_partial(items[first:first + cnt], r, first)
                    assert parts[288 * rank: 288 * rank + 288] == want, (cfg, world, rank)
                assert ok is True, (cfg, world)


# ------------------------------------------------------------------ b. forged pairs
# (name, pair, options, simulated ranks of the phase entry points)
PLACEMENTS = [
    ("neighbours", (0, 1), {}, 1),                                 # every weight equal
    ("one_rlc_block_apart", (5, 133), {}, 1),                      # exponent local to a 128-thread block
    ("one_chunk_apart", (7, 57), {"chunk_blobs": 50}, 1),          # exponent restarting at each chunk
    ("one_super_batch_apart", (11, 111), {"verify_super_blobs": 100}, 1),   # ... at each staging super-batch
    ("same_local_index_world2", (3, 153), {}, 2),                  # `first` ignored
    ("same_local_index_world3", (104, 204), {}, 3),
]


def _check_forgery(lw, s, bt, coms, proofs, forged, world, what):
    for name, fn in entry_points(world).items():
        assert fn(lw, s, bt, coms, proofs) is True, (what, name, "valid batch")
        assert fn(lw, s, bt, coms, forged) is False, (what, name, "forged pair accepted")


@pytest.mark.parametrize("name,pair,opts,world", PLACEMENTS, ids=[p[0] for p in PLACEMENTS])
def test_forged_pair_is_rejected(lw, env, name, pair, opts, world):
    i, j = pair
    if world > 1:   # the pair sits at the same local index of two ranks
        shards = [lw.shard_range(N, world, r) for r in range(world)]
        fi, fj = (next(f for f, c in shards if f <= k < f + c) for k in pair)
        assert fi != fj and i - fi == j - fj
    blobs, coms, proofs = cols(env.items)
    forged = _forge.forge_blob_batch(env.o, blobs, coms, proofs, i, j)
    with options(lw, **opts):
        _check_forgery(lw, env.s, Batch(blobs), coms, proofs, forged, world, name)


def test_forged_pair_among_identical_items(lw, env):
    """N copies of one item: equal points meet in one bucket of the variable-base MSMs."""
    blobs, coms, proofs = cols([env.items[0]] * N)
    forged = _forge.forge_blob_batch(env.o, blobs, coms, proofs, 3, 170)
    _check_forgery(lw, env.s, Batch(blobs), coms, proofs, forged, 2, "identical items")


@pytest.mark.parametrize("env", [0], indirect=True, ids=["ref"])
def test_forged_pair_in_a_4096_blob_batch(lw, env):
    """The benchmarked configuration: 4096 blobs at the default verification options, the pair at both ends."""
    n = 4096
    blobs = [lw.synth_blob_host(k) for k in range(n)]
    coms, proofs, st = lw.commit_and_prove_batch(b"".join(blobs), n, env.s)
    assert st == [0] * n
    for k in (0, n - 1):
        assert coms[k] == env.o.blob_to_kzg_commitment(blobs[k]) and proofs[k] == env.o.compute_blob_kzg_proof(blobs[k], coms[k])
    forged = _forge.forge_blob_batch(env.o, blobs, coms, proofs, 0, n - 1)
    _check_forgery(lw, env.s, Batch(blobs), coms, proofs, forged, 2, "4096 blobs")


# ------------------------------------------------------------------ c. points outside G1
@pytest.mark.parametrize("split", [0, 1], ids=["inline", "split"])
@pytest.mark.parametrize("n", [1, 2, 65, 300])
def test_points_outside_g1_are_rejected(lw, env, n, split):
    """The decompression kernel, the separate subgroup kernels (verify_split_subgroup = 1 and n > 64) and the deferred
    check of single verification (n = 1) must all report the point; the next valid call must verify."""
    code = _forge.decode_error_code(env.mode)
    blobs, coms, proofs = cols(env.items[:n])
    bt = Batch(blobs)
    calls = {
        "host": v_host,
        "device": v_device,
        "phase1": lambda lw, s, bt, c, p: lw.verify_batch_phase1(bt.flat, b"".join(c), b"".join(p), bt.n, s),
    }
    good = {"host": v_host, "device": v_device, "phase1": lambda lw, s, bt, c, p: run_phases(lw, s, bt, c, p, 1, False)[0]}
    with options(lw, verify_split_subgroup=split):
        for enc in _forge.non_g1_points():
            for pos in sorted({0, n // 2, n - 1}):
                for role in ("commitment", "proof"):
                    c2, p2 = list(coms), list(proofs)
                    (c2 if role == "commitment" else p2)[pos] = enc
                    for name, fn in calls.items():
                        with pytest.raises(lw.KzgError) as e:
                            fn(lw, env.s, bt, c2, p2)
                        assert e.value.code == code, (name, role, pos)
                        assert good[name](lw, env.s, bt, coms, proofs) is True, (name, role, pos, "valid batch after a rejected one")


# ------------------------------------------------------------------ d. cells
def test_forged_cell_pairs(lw, env, py_setup):
    co = cells.CellOracle(py_setup, env.mode)
    tau = py_setup.tau
    blobs = [env.items[0].blob, env.items[1].blob]
    coms = [env.items[0].commitment, env.items[1].commitment]
    cl, pl = {}, {}
    for b, blob in enumerate(blobs):
        cs, ps = lw.compute_cells_and_kzg_proofs(blob, env.s)
        for k in range(128):
            cl[b, k], pl[b, k] = cs[k], ps[k]
    cases = [
        ("two cells of one blob", [(0, 3), (0, 9), (0, 70), (1, 5)], 1, 2),
        ("one cell index, two blobs", [(0, 9), (1, 9), (0, 3)], 0, 1),
        ("positions 5 and 133 of 256", [(b, k) for b in range(2) for k in range(128)], 5, 133),
    ]
    for name, sel, i, j in cases:
        c = [coms[b] for b, _ in sel]
        idx = [k for _, k in sel]
        cel = [cl[x] for x in sel]
        prf = [pl[x] for x in sel]
        forged = _forge.forge_cell_batch(tau, idx, prf, i, j)
        assert lw.verify_cell_kzg_proof_batch(c, idx, cel, prf, env.s) is True, name
        assert lw.verify_cell_kzg_proof_batch(c, idx, cel, forged, env.s) is False, name
        assert co.verify_cell_kzg_proof_batch(c, idx, cel, forged) is False, name
        assert _forge.weighted_cell_check(co, c, idx, cel, forged, [1] * len(sel)) is True, name
    for enc in _forge.non_g1_points():
        with pytest.raises(lw.KzgError) as e:
            lw.verify_cell_kzg_proof_batch([coms[0], coms[1]], [3, 9], [cl[0, 3], cl[1, 9]], [pl[0, 3], enc], env.s)
        assert e.value.code == co.bad
        assert lw.verify_cell_kzg_proof_batch([coms[0], coms[1]], [3, 9], [cl[0, 3], cl[1, 9]], [pl[0, 3], pl[1, 9]], env.s) is True
