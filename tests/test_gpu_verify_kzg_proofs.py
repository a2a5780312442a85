"""GPU tier: n independent single-opening checks per call, lwkzg_verify_kzg_proofs[_device] (include/lwkzg.h part 2).

Every item must get exactly what verify_kzg_proof returns for it alone (verdict and error code), in modes 0, 1 and 2,
whatever the other items of its warp are; and each verdict must come from the item's own pairing check, not from an
aggregate over the call."""
import ctypes
import os
import random

import pytest

from oracle.py import bls, kzg
from tests import _forge
from tests.golden.make_cell_fixtures import make_blob

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
R = bls.R
P = bls.P
PASS = 32768   # items per pass (VP_PASS in csrc/lwkzg.cu)
INF = b"\xc0" + bytes(47)


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
    """Openings of one mode, by kind: each kind is a (commitment, z, y, proof) tuple."""

    def __init__(self, lw, s, mode, py_setup):
        self.lw, self.s, self.mode = lw, s, mode
        self.o = _forge.oracle_for(mode, py_setup)
        fe = lambda v: _forge.fe_bytes(mode, v)   # noqa: E731
        rnd = random.Random(4844 + mode)
        nb = 4
        blobs = [make_blob(700 + b, mode) for b in range(nb)]
        zero_blob = bytes(4096 * 32)
        const = 0xC0FFEE
        const_blob = (fe(const) * 4096) if mode != 0 else fe(const) + bytes(4095 * 32)
        blobs += [zero_blob, const_blob, blobs[0]]
        zs = [rnd.randrange(R) for _ in range(nb)] + [rnd.randrange(R), rnd.randrange(R), 0]
        coms, st = lw.blob_to_kzg_commitment_batch(b"".join(blobs), len(blobs), s)
        assert st == [0] * len(blobs)
        proofs, ys, st = lw.compute_kzg_proof_batch(b"".join(blobs), b"".join(fe(z) for z in zs), len(blobs), s)
        assert st == [0] * len(blobs)
        assert coms[4] == INF and proofs[5] == INF and proofs[4] == INF
        yv = [int.from_bytes(y, "little" if mode == 1 else "big") for y in ys]
        assert max(yv[:nb]).bit_length() > 248   # full-length y
        self.valid = [(coms[i], fe(zs[i]), ys[i], proofs[i]) for i in range(len(blobs))]
        self.zs, self.yv = zs, yv
        c0, z0, y0, p0 = self.valid[0]
        c1, z1, y1, p1 = self.valid[1]
        bad = _forge.non_g1_points()
        k = {
            "true": self.valid[0], "true1": self.valid[1], "true2": self.valid[2], "true3": self.valid[3],
            "zero_blob": self.valid[4], "const_poly": self.valid[5], "z_zero": self.valid[6],
            "wrong_y": (c0, z0, fe(yv[0] + 1), p0), "wrong_z": (c0, fe(zs[0] + 1), y0, p0),
            "swapped_a": (c0, z0, y0, p1), "swapped_b": (c1, z1, y1, p0), "y_zero": (c0, z0, fe(0), p0),
            "bad_flag": (bytes([c0[0] & 0x7F]) + c0[1:], z0, y0, p0),
            "bad_inf": (bytes([0xC0]) + bytes(46) + b"\x01", z0, y0, p0),
            "x_ge_p": (bytes([0x80 | ((P + 3) >> 376)]) + (P + 3).to_bytes(48, "big")[1:], z0, y0, p0),
            "off_curve_c": (_off_curve(), z0, y0, p0), "off_curve_pi": (c0, z0, y0, _off_curve()),
            "non_g1_c": (bad[0], z0, y0, p0), "non_g1_c2": (bad[1], z0, y0, p0),
            "non_g1_pi": (c0, z0, y0, bad[0]), "non_g1_pi2": (c0, z0, y0, bad[1]),
            "pi_inf_wrong": (c0, z0, y0, INF), "c_inf_wrong": (INF, z0, y0, p0),
        }
        big = (1 << 256) - 1
        enc = "little" if mode == 1 else "big"
        k["z_is_r"] = (c0, R.to_bytes(32, enc), y0, p0)
        k["y_is_r"] = (c0, z0, R.to_bytes(32, enc), p0)
        k["z_max"] = (c0, big.to_bytes(32, enc), y0, p0)
        k["y_r_plus"] = (c0, z0, (R + yv[0]).to_bytes(32, enc), p0)
        self.kinds = k
        self.expect = {name: self.single(it) for name, it in k.items()}

    def single(self, item):
        """(verdict, code) of one verify_kzg_proof call"""
        try:
            return self.lw.verify_kzg_proof(*item, self.s), 0
        except self.lw.KzgError as e:
            return False, e.code

    def run(self, items):
        return self.lw.verify_kzg_proofs([i[0] for i in items], [i[1] for i in items], [i[2] for i in items], [i[3] for i in items], self.s)


@pytest.fixture(scope="module", params=[0, 1, 2], ids=["mode0", "mode1", "mode2"])
def data(request, lw, py_setup):
    s = _load(lw, request.param)
    yield Data(lw, s, request.param, py_setup)
    s.free()


def _oracle(o, item):
    try:
        return bool(o.verify_kzg_proof(*item)), 0
    except kzg.KzgError as e:
        return False, e.code


def test_kinds_match_single_call_and_oracle(data):
    names = list(data.kinds)
    ok, st = data.run([data.kinds[n] for n in names])
    for i, n in enumerate(names):
        assert (ok[i], st[i]) == data.expect[n], n
        assert _oracle(data.o, data.kinds[n]) == data.expect[n], n
    e = data.expect
    for n in ("true", "true1", "true2", "true3", "zero_blob", "const_poly", "z_zero"):
        assert e[n] == (True, 0), n
    for n in ("wrong_y", "wrong_z", "swapped_a", "swapped_b", "y_zero", "pi_inf_wrong", "c_inf_wrong"):
        assert e[n] == (False, 0), n
    code = _forge.decode_error_code(data.mode)
    for n in ("bad_flag", "off_curve_c", "off_curve_pi", "non_g1_c", "non_g1_c2", "non_g1_pi", "non_g1_pi2"):
        assert e[n] == (False, code), n
    for n in ("z_is_r", "y_is_r", "z_max", "y_r_plus"):
        assert e[n] == ((False, 1) if data.mode else e[n]), n
    if data.mode:
        assert e["bad_inf"] == (False, 1) and e["x_ge_p"] == (False, 1)
    else:
        assert e["y_r_plus"] == (True, 0)   # mode 0 reduces y mod r


def _layout(data, names, n):
    items = [data.kinds[names[i % len(names)]] for i in range(n)]
    want = [data.expect[names[i % len(names)]] for i in range(n)]
    ok, st = data.run(items)
    got = list(zip(ok, st))
    bad = [i for i in range(n) if got[i] != want[i]]
    assert not bad, [(i, names[i % len(names)], got[i], want[i]) for i in bad[:8]]


def test_every_kind_at_many_lanes_with_ragged_tail(data):
    # 29 kinds cycling over 4 full 64-thread blocks and a partial last one: every kind lands at several lanes of one
    # warp, next to every other kind, and in the partial last warp
    _layout(data, list(data.kinds), 64 * 4 + 45)


def test_valid_and_invalid_alternate_lane_by_lane(data):
    _layout(data, ["true", "non_g1_pi", "const_poly", "bad_flag", "zero_blob", "non_g1_c", "true1", "off_curve_c"], 96 + 7)
    _layout(data, ["true", "pi_inf_wrong", "true1", "c_inf_wrong", "const_poly", "wrong_y"], 70)


def test_forged_pair_fails_item_by_item(data):
    """A pair that cancels under equal weights (it can pass a weighted aggregate check) is rejected item by item."""
    tau = data.o.s.tau
    (c0, z0, y0, p0), (c1, z1, y1, p1) = data.valid[0], data.valid[1]
    f0, f1 = _forge.forge_pair(p0, p1, (tau - data.zs[0]) % R, (tau - data.zs[1]) % R)
    # with equal weights the two changes cancel: sum over the pair of (C - yG - (tau - z) pi) stays the point at infinity
    d = [(tau - data.zs[0]) % R, (tau - data.zs[1]) % R]
    moved = bls.g1_add(bls.g1_mul(bls.g1_add(bls.g1_decompress(f0), bls.g1_neg(bls.g1_decompress(p0))), d[0]),
                       bls.g1_mul(bls.g1_add(bls.g1_decompress(f1), bls.g1_neg(bls.g1_decompress(p1))), d[1]))
    assert moved is None or moved == bls.g1_mul(bls.G1, 0)
    items = [(c0, z0, y0, f0), (c1, z1, y1, f1), data.valid[2]]
    ok, st = data.run(items)
    assert ok == [False, False, True] and st == [0, 0, 0]
    assert data.single(items[0]) == (False, 0) and data.single(items[1]) == (False, 0)


def _tiled(data, n):
    names = ["true", "wrong_y", "non_g1_pi", "const_poly", "y_is_r", "zero_blob", "true2", "bad_flag", "swapped_a"]
    items = [data.kinds[names[i % len(names)]] for i in range(n)]
    want = [data.expect[names[i % len(names)]] for i in range(n)]
    return items, want


def test_several_passes_host_and_device(data, lw):
    import torch

    n = 2 * PASS + 77
    items, want = _tiled(data, n)
    ok, st = data.run(items)
    assert list(zip(ok, st)) == want
    dev = torch.device("cuda", 0)
    cols = [torch.frombuffer(bytearray(b"".join(it[k] for it in items)), dtype=torch.uint8).to(dev) for k in range(4)]
    d_ok = torch.full((n,), 7, dtype=torch.int32, device=dev)
    d_st = torch.full((n,), 7, dtype=torch.int32, device=dev)
    lw.verify_kzg_proofs_device(d_ok.data_ptr(), cols[0].data_ptr(), cols[1].data_ptr(), cols[2].data_ptr(), cols[3].data_ptr(), n, data.s, 0,
                                d_st.data_ptr())
    torch.cuda.synchronize()
    assert d_ok.cpu().tolist() == [int(v) for v in ok]
    assert d_st.cpu().tolist() == st


def test_device_form_on_a_stream_without_status(data, lw):
    import torch

    names = list(data.kinds)
    n = 3 * 64 + 11
    items = [data.kinds[names[(i * 7) % len(names)]] for i in range(n)]
    ok, st = data.run(items)
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(stream):
        cols = [torch.frombuffer(bytearray(b"".join(it[k] for it in items)), dtype=torch.uint8).to(dev, non_blocking=False) for k in range(4)]
        d_ok = torch.full((n,), 7, dtype=torch.int32, device=dev)
        torch.cuda._sleep(50_000_000)   # the call must wait for earlier work on its stream
        lw.verify_kzg_proofs_device(d_ok.data_ptr(), cols[0].data_ptr(), cols[1].data_ptr(), cols[2].data_ptr(), cols[3].data_ptr(), n, data.s,
                                    stream.cuda_stream, 0)
        out = d_ok.to("cpu", non_blocking=False)
    stream.synchronize()
    assert out.numpy().astype("int32").tobytes() == b"".join(int(v).to_bytes(4, "little") for v in ok)


def test_whole_call_errors(data, lw):
    lib = lw.load_library()
    sp = lw.api._sp(data.s)
    c, z, y, p = data.kinds["true"]
    assert lib.lwkzg_verify_kzg_proofs(None, None, None, None, None, 0, sp, None) == 0
    assert lib.lwkzg_verify_kzg_proofs_device(None, None, None, None, None, 0, sp, None, None) == 0
    ok = (ctypes.c_bool * 1)()
    assert lib.lwkzg_verify_kzg_proofs(None, c, z, y, p, 1, sp, None) == 1
    assert lib.lwkzg_verify_kzg_proofs(ok, None, z, y, p, 1, sp, None) == 1
    assert lib.lwkzg_verify_kzg_proofs(ok, c, z, None, p, 1, sp, None) == 1
    assert lib.lwkzg_verify_kzg_proofs_device(None, 16, 16, 16, 16, 1, sp, None, None) == 1
    # status == NULL: the first failing item's code, every verdict still written
    names = ["true", "wrong_y", "non_g1_pi", "true1", "y_is_r"]
    items = [data.kinds[n] for n in names]
    oks = (ctypes.c_bool * 5)()
    rc = lib.lwkzg_verify_kzg_proofs(oks, b"".join(i[0] for i in items), b"".join(i[1] for i in items), b"".join(i[2] for i in items),
                                     b"".join(i[3] for i in items), 5, sp, None)
    assert rc == _forge.decode_error_code(data.mode)
    assert list(oks) == [data.expect[n][0] for n in names]
    rc = lib.lwkzg_verify_kzg_proofs(oks, items[0][0] + items[3][0], items[0][1] + items[3][1], items[0][2] + items[3][2], items[0][3] + items[3][3],
                                     2, sp, None)
    assert rc == 0 and list(oks)[:2] == [True, True]


def test_two_gpus_match_one(data, lw):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    items, want = _tiled(data, 4 * 64 + 3)
    one = data.run(items)
    lw.set_devices([0, 1])
    try:
        two = data.run(items)
    finally:
        lw.set_devices([])
    assert two == one and list(zip(*one)) == want
