"""GPU tier: many independent blob-proof batches per call, lwkzg_verify_blob_kzg_proof_batches[_device] (include/lwkzg.h
part 2).

Every batch must get exactly what ONE verify_blob_kzg_proof_batch call over that batch alone returns (verdict and error
code), in modes 0, 1 and 2, whatever its neighbours are: its own challenge over its own tuples, its own weights
r_b^0 .. r_b^(n_b - 1), its own failures."""
import ctypes
import os

import pytest

from oracle.py import bls
from tests import _forge
from tests.golden.make_cell_fixtures import make_blob

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
R = bls.R
P = bls.P
BLOB = 4096 * 32


@pytest.fixture(scope="module")
def lw():
    import lambdaworks_kzg_b200 as m

    m.load_library()
    return m


def _load(lw, mode):
    lw.set_option("mode", mode)
    lw.set_option("window_bits", 8)
    try:
        return lw.load_trusted_setup_file(os.path.join(GOLDEN, "trusted_setup.txt"))
    finally:
        lw.set_option("mode", 0)
        lw.set_option("window_bits", 16)


def _off_curve() -> bytes:
    for x in range(1, 100):
        if pow((x ** 3 + 4) % P, (P - 1) // 2, P) == P - 1:
            return bytes([0x80]) + x.to_bytes(48, "big")[1:]
    raise AssertionError("no x without a square root")


class Data:
    """Items (blob, commitment, proof) of one mode: valid ones, and by kind the invalid ones."""

    def __init__(self, lw, s, mode, py_setup):
        self.lw, self.s, self.mode = lw, s, mode
        self.o = _forge.oracle_for(mode, py_setup)
        fe = lambda v: _forge.fe_bytes(mode, v)   # noqa: E731
        blobs = [make_blob(900 + 17 * mode + b, mode) for b in range(8)]
        const = 0xC0FFEE
        blobs.append(bytes(BLOB))   # zero blob: commitment and proof at infinity
        blobs.append((fe(const) * 4096) if mode != 0 else fe(const) + bytes(4095 * 32))   # constant polynomial: proof at infinity
        coms, proofs, st = lw.commit_and_prove_batch(b"".join(blobs), len(blobs), s)
        assert st == [0] * len(blobs)
        inf = b"\xc0" + bytes(47)
        assert coms[8] == inf and proofs[8] == inf and proofs[9] == inf
        self.valid = list(zip(blobs, coms, proofs))
        b0, c0, p0 = self.valid[0]
        b1, c1, p1 = self.valid[1]
        g1bad = _forge.non_g1_points()
        self.invalid = {
            "bad_encoding_c": (b0, b"\x00" * 47 + b"\x01", p0),
            "bad_encoding_pi": (b0, c0, b"\x00" * 47 + b"\x02"),
            "off_curve_c": (b0, _off_curve(), p0),
            "off_curve_pi": (b0, c0, _off_curve()),
            "non_g1_c": (b0, g1bad[0], p0),
            "non_g1_pi": (b0, c0, g1bad[1]),
        }
        if mode:   # a blob word >= r: reduced in mode 0, rejected by the c-kzg modes
            word = R.to_bytes(32, "little" if mode == 1 else "big")
            self.invalid["blob_word_r"] = (word + b1[32:], c1, p1)
        self.code = _forge.decode_error_code(mode)

    def item(self, k):
        return self.valid[k % len(self.valid)]

    def single(self, batch):
        """(verdict, code) of one verify_blob_kzg_proof_batch call over the batch"""
        try:
            return self.lw.verify_blob_kzg_proof_batch([i[0] for i in batch], [i[1] for i in batch], [i[2] for i in batch], self.s), 0
        except self.lw.KzgError as e:
            return False, e.code

    def single_blob(self, it):
        try:
            return self.lw.verify_blob_kzg_proof(it[0], it[1], it[2], self.s), 0
        except self.lw.KzgError as e:
            return False, e.code

    def run(self, batches):
        return self.lw.verify_blob_kzg_proof_batches([([i[0] for i in b], [i[1] for i in b], [i[2] for i in b]) for b in batches], self.s)

    def check(self, batches):
        ok, st = self.run(batches)
        got = list(zip(ok, st))
        want = [self.single(b) for b in batches]
        bad = [(k, len(batches[k]), got[k], want[k]) for k in range(len(batches)) if got[k] != want[k]]
        assert not bad, bad
        return got


@pytest.fixture(scope="module", params=[0, 1, 2], ids=["mode0", "mode1", "mode2"])
def data(request, lw, py_setup):
    s = _load(lw, request.param)
    yield Data(lw, s, request.param, py_setup)
    s.free()


def _mixed(d):
    """Empty, one-blob, 2-, 6- and ~100-blob batches, the zero blob and a constant polynomial, wrong and swapped proofs and
    a commitment of another blob."""
    v = d.valid
    (b0, c0, p0), (b1, c1, p1), (b3, c3, p3), (b4, c4, p4) = v[0], v[1], v[3], v[4]
    big = [d.item(k) for k in range(101)]
    big_bad = list(big)
    big_bad[57] = (big[57][0], big[57][1], big[58][2])
    return [
        [],
        [v[2]],
        [v[0], v[1]],
        [d.item(k) for k in range(2, 8)],
        [(b0, c0, p1)],                               # one blob, wrong proof
        [(b0, c0, p1), (b1, c1, p0)],                 # swapped proofs
        [v[5], v[6], (b3, c4, p3), v[7], v[2], v[9]],  # a commitment of another blob
        big,
        [v[8], v[9]],                                 # zero blob, constant polynomial
        [],
        [v[9]],
        [v[8]],
        big_bad,
        [(b4, c4, p4), (b3, c3, p3)],
    ]


def test_matches_single_calls_and_oracle(data):
    batches = _mixed(data)
    got = data.check(batches)
    empty = (data.mode != 0, 0)
    assert got[0] == empty and got[9] == empty
    assert [g[0] for g in got] == [empty[0], True, True, True, False, False, False, True, True, empty[0], True, True, False, True]
    assert all(g[1] == 0 for g in got)
    for k, b in enumerate(batches):   # one blob: verify_blob_kzg_proof's verdict
        if len(b) == 1:
            assert got[k] == data.single_blob(b[0]), k
    for k in (2, 5, 8, 10):   # a sample against the oracle
        b = batches[k]
        assert bool(data.o.verify_blob_kzg_proof_batch([i[0] for i in b], [i[1] for i in b], [i[2] for i in b])) == got[k][0], k


def test_invalid_items_fail_only_their_batch(data):
    v = data.valid
    for name, bad in data.invalid.items():
        batches = [
            [bad, v[1], v[2], v[3], v[4]],          # first position
            [v[1], v[2]],
            [v[1], v[2], bad, v[3], v[4]],          # middle
            [v[5], v[6], v[7], v[3], bad],          # last
            [bad],                                  # adjacent failing batches
            [v[0], bad],
            [v[3], v[4], v[5]],
        ]
        got = data.check(batches)
        assert got == [(False, data.code), (True, 0), (False, data.code), (False, data.code), (False, data.code), (False, data.code), (True, 0)], name


def _forged(d, idx, i, j):
    items = [d.item(k) for k in idx]
    proofs = _forge.forge_blob_batch(d.o, [t[0] for t in items], [t[1] for t in items], [t[2] for t in items], i, j)
    return [(t[0], t[1], p) for t, p in zip(items, proofs)]


def test_forged_pair_needs_its_batch_weights(data, lw):
    """A pair that passes exactly when its two weights are equal fails its batch; the honest batch beside it passes."""
    forged = _forged(data, [0, 1, 2], 0, 1)
    honest = [data.item(k) for k in (3, 4, 5)]
    assert _forge.weighted_batch_check(data.o, [t[0] for t in forged], [t[1] for t in forged], [t[2] for t in forged], [1, 1, 1])
    assert data.check([honest, forged, honest]) == [(True, 0), (False, 0), (True, 0)]
    # a pass of at most 4 blobs: the forged batch right after a pass boundary, and a forged pair straddling the staging
    # boundary of a 6-blob batch larger than a pass
    big = _forged(data, [2, 3, 4, 5, 6, 7], 3, 4)
    old = lw.get_option("verify_super_blobs")
    lw.set_option("verify_super_blobs", 4)
    try:
        got = data.check([honest, forged, big, honest[:2]])
    finally:
        lw.set_option("verify_super_blobs", old)
    assert got == [(True, 0), (False, 0), (False, 0), (True, 0)]


def test_challenges_per_batch(data, lw):
    batches = [[], [data.item(0)], [data.item(1), data.item(2)], [data.item(k) for k in (3, 4, 5, 6, 7, 9)], [data.item(8), data.item(0)]]
    data.run(batches)
    rs = lw.debug_blob_batch_challenges(len(batches), data.s)
    assert rs[0] == 0 and rs[1] == 0
    for k in (2, 3, 4):
        b = batches[k]
        zs = [_forge.challenge(data.o, t[0], t[1]) for t in b]
        ys = [_forge.poly_at(data.o, t[0], z) for t, z in zip(b, zs)]
        assert rs[k] == _forge.batch_challenge(data.mode, [t[1] for t in b], zs, ys, [t[2] for t in b]), k
    assert len(set(rs[2:])) == 3


def test_passes_match_default(data, lw):
    batches = _mixed(data)
    default = data.run(batches)
    old = lw.get_option("verify_super_blobs")
    lw.set_option("verify_super_blobs", 5)
    try:
        small = data.run(batches)
        d = _device_run(data, lw, batches, with_status=True)
    finally:
        lw.set_option("verify_super_blobs", old)
    assert small == default
    assert d == ([int(v) for v in default[0]], default[1])


def _flat(batches):
    items = [t for b in batches for t in b]
    offsets = [0]
    for b in batches:
        offsets.append(offsets[-1] + len(b))
    return items, offsets


def _device_run(data, lw, batches, with_status, stream=None):
    import torch

    items, offsets = _flat(batches)
    k = len(batches)
    dev = torch.device("cuda", 0)
    cols = [torch.frombuffer(bytearray(b"".join(t[c] for t in items) or b"\0"), dtype=torch.uint8).to(dev) for c in range(3)]
    d_ok = torch.full((k,), 7, dtype=torch.int32, device=dev)
    d_st = torch.full((k,), 7, dtype=torch.int32, device=dev)
    lw.verify_blob_kzg_proof_batches_device(d_ok.data_ptr(), cols[0].data_ptr(), cols[1].data_ptr(), cols[2].data_ptr(), offsets, data.s,
                                            stream or 0, d_st.data_ptr() if with_status else 0)
    torch.cuda.synchronize()
    return d_ok.cpu().tolist(), (d_st.cpu().tolist() if with_status else None)


def test_device_form(data, lw):
    import torch

    batches = _mixed(data)[:9] + [[data.invalid["non_g1_pi"], data.item(1)], [data.item(2)]]
    ok, st = data.run(batches)
    assert _device_run(data, lw, batches, True) == ([int(v) for v in ok], st)
    assert _device_run(data, lw, batches, False)[0] == [int(v) for v in ok]
    # on a non-default stream, inputs written by work queued on that stream just before the call
    items, offsets = _flat(batches)
    dev = torch.device("cuda", 0)
    src = [torch.frombuffer(bytearray(b"".join(t[c] for t in items)), dtype=torch.uint8).to(dev) for c in range(3)]
    torch.cuda.synchronize()
    stream = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(stream):
        dst = [torch.zeros_like(x) for x in src]
        d_ok = torch.full((len(batches),), 7, dtype=torch.int32, device=dev)
        torch.cuda._sleep(50_000_000)
        for x, y in zip(dst, src):
            x.copy_(y)
        lw.verify_blob_kzg_proof_batches_device(d_ok.data_ptr(), dst[0].data_ptr(), dst[1].data_ptr(), dst[2].data_ptr(), offsets, data.s,
                                                stream.cuda_stream, 0)
        out = d_ok.to("cpu", non_blocking=False)
    stream.synchronize()
    assert out.tolist() == [int(v) for v in ok]
    # the challenges of the device call
    rs = lw.debug_blob_batch_challenges(len(batches), data.s)
    assert rs[0] == 0 and rs[1] == 0 and rs[2] != 0


def test_host_form_from_pinned_memory(data, lw):
    import torch

    batches = _mixed(data)
    ok, st = data.run(batches)   # Python bytes: pageable, staged through the pinned ring (the 101-blob batch is > 4 MiB)
    items, offsets = _flat(batches)
    pinned = [torch.frombuffer(bytearray(b"".join(t[c] for t in items)), dtype=torch.uint8).pin_memory() for c in range(3)]
    k = len(batches)
    off = (ctypes.c_uint64 * (k + 1))(*offsets)
    oks = (ctypes.c_bool * k)()
    sts = (ctypes.c_int * k)()
    rc = lw.load_library().lwkzg_verify_blob_kzg_proof_batches(oks, pinned[0].data_ptr(), pinned[1].data_ptr(), pinned[2].data_ptr(), off, k,
                                                               lw.api._sp(data.s), sts)
    assert rc == 0 and list(oks) == ok and list(sts) == st


def test_whole_call_errors(data, lw):
    lib = lw.load_library()
    sp = lw.api._sp(data.s)
    b, c, p = data.item(0)
    ok = (ctypes.c_bool * 4)()
    st = (ctypes.c_int * 4)()
    U = ctypes.c_uint64
    assert lib.lwkzg_verify_blob_kzg_proof_batches(None, None, None, None, None, 0, sp, None) == 0
    assert lib.lwkzg_verify_blob_kzg_proof_batches_device(None, None, None, None, None, 0, sp, None, None) == 0
    one = (U * 2)(0, 1)
    assert lib.lwkzg_verify_blob_kzg_proof_batches(None, b, c, p, one, 1, sp, None) == 1
    assert lib.lwkzg_verify_blob_kzg_proof_batches(ok, b, c, p, None, 1, sp, None) == 1
    assert lib.lwkzg_verify_blob_kzg_proof_batches(ok, None, c, p, one, 1, sp, None) == 1
    assert lib.lwkzg_verify_blob_kzg_proof_batches(ok, b, c, None, one, 1, sp, None) == 1
    assert lib.lwkzg_verify_blob_kzg_proof_batches(ok, b, c, p, (U * 2)(1, 1), 1, sp, None) == 1       # offsets[0] != 0
    assert lib.lwkzg_verify_blob_kzg_proof_batches(ok, b, c, p, (U * 3)(0, 1, 0), 2, sp, None) == 1    # decreasing
    assert lib.lwkzg_verify_blob_kzg_proof_batches(ok, b, c, p, (U * 2)(0, (1 << 24) + 1), 1, sp, None) == 1
    assert lib.lwkzg_verify_blob_kzg_proof_batches_device(None, 16, 16, 16, one, 1, sp, None, None) == 1
    assert lib.lwkzg_verify_blob_kzg_proof_batches_device(16, None, 16, 16, one, 1, sp, None, None) == 1
    assert lib.lwkzg_verify_blob_kzg_proof_batches_device(16, 16, 16, 16, None, 1, sp, None, None) == 1
    assert lib.lwkzg_verify_blob_kzg_proof_batches_device(16, 16, 16, 16, (U * 2)(1, 1), 1, sp, None, None) == 1
    assert lib.lwkzg_verify_blob_kzg_proof_batches_device(16, 16, 16, 16, (U * 3)(0, 1, 0), 2, sp, None, None) == 1
    # only empty batches: NULL inputs are fine, every batch gets the mode's empty verdict
    assert lib.lwkzg_verify_blob_kzg_proof_batches(ok, None, None, None, (U * 3)(0, 0, 0), 2, sp, st) == 0
    assert list(ok)[:2] == [data.mode != 0] * 2 and list(st)[:2] == [0, 0]
    # status == NULL: the first failing batch's code, every verdict still written
    bad = data.invalid["non_g1_c"]
    batches = [[data.item(0), data.item(1)], [data.item(2), bad], [(b, c, data.item(1)[2])], [data.item(3)]]
    items, offsets = _flat(batches)
    rc = lib.lwkzg_verify_blob_kzg_proof_batches(ok, b"".join(t[0] for t in items), b"".join(t[1] for t in items), b"".join(t[2] for t in items),
                                                 (U * 5)(*offsets), 4, sp, None)
    assert rc == data.code and list(ok) == [True, False, False, True]


def test_two_gpus_match_one(data, lw):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    batches = _mixed(data)
    one = data.run(batches)
    rs1 = lw.debug_blob_batch_challenges(len(batches), data.s)
    lw.set_devices([0, 1])
    try:
        two = data.run(batches)
        rs2 = lw.debug_blob_batch_challenges(len(batches), data.s)
    finally:
        lw.set_devices([])
    assert two == one and rs2 == rs1


def test_mode0_one_blob_batch_subtracts_g1_values_0(lw, py_setup):
    """MODE_REFERENCE on a setup of k tau^i G (G2 points unchanged, so g1_values[0] = kG is not the generator): an honest
    one-blob batch passes, as verify_blob_kzg_proof does (it subtracts y g1_values[0]); an honest two-blob batch with
    y != 0 fails, as verify_blob_kzg_proof_batch does (it subtracts y G)."""
    k = 7
    pts = b"".join(x.to_bytes(48, "big") + y.to_bytes(48, "big") for x, y in py_setup.g1)
    g1 = b"".join(lw.g1_lincomb(pts[96 * i: 96 * i + 96], k.to_bytes(32, "big"), 1) for i in range(len(py_setup.g1)))
    lines = open(os.path.join(GOLDEN, "trusted_setup.txt")).read().split()
    n1, n2 = int(lines[0]), int(lines[1])
    g2 = b"".join(bytes.fromhex(h) for h in lines[2 + n1: 2 + n1 + n2])
    assert g1[:48] == bls.g1_compress(bls.g1_mul(bls.G1, k))
    lw.set_option("window_bits", 8)
    try:
        s = lw.load_trusted_setup(g1, g2)
    finally:
        lw.set_option("window_bits", 16)
    try:
        blobs = [make_blob(4242 + i, 0) for i in range(2)]
        coms, proofs, st = lw.commit_and_prove_batch(b"".join(blobs), 2, s)
        assert st == [0, 0]
        items = list(zip(blobs, coms, proofs))
        batches = [[items[0]], items, [items[1]]]
        want = [(True, 0), (False, 0), (True, 0)]
        for b, w in zip(batches, want):
            assert lw.verify_blob_kzg_proof_batch([t[0] for t in b], [t[1] for t in b], [t[2] for t in b], s) == w[0]
        assert lw.verify_blob_kzg_proof(*items[0], s) is True
        ok, st = lw.verify_blob_kzg_proof_batches([([t[0] for t in b], [t[1] for t in b], [t[2] for t in b]) for b in batches], s)
        assert list(zip(ok, st)) == want
    finally:
        s.free()
