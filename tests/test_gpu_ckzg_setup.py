"""GPU tier: c-kzg-4844 trusted setups (lwkzg_load_trusted_setup[_file]_ckzg) over the tau = 1337 golden setup.

The c-kzg file is built at test time: its Lagrange section from mode-1 settings of tests/golden/trusted_setup.txt
(un-bit-reversed, pinned against [l_k(tau)]G), its G2 and monomial sections from the golden file.  The new loaders
must give the settings load_trusted_setup_file gives for the golden file in every mode, and reject every setup whose
sections are not one powers-of-tau."""
import ctypes
import hashlib
import json
import os
import random
import tempfile

import pytest

from tests._ckzg_setup import GOLDEN, N, bitrev12, forged_g2_outside_subgroup, golden_sections, lagrange_from_settings, lagrange_scalar, write_text
from tests.golden.make_cell_fixtures import make_blob

pytestmark = pytest.mark.gpu

SETUP = os.path.join(GOLDEN, "trusted_setup.txt")
R = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001


@pytest.fixture(scope="module")
def lw():
    import lambdaworks_kzg_b200 as m

    m.load_library()
    m.set_option("window_bits", 8)
    m.set_option("cell_window_bits", 8)
    yield m
    m.set_option("window_bits", 16)
    m.set_option("cell_window_bits", 13)
    m.set_option("mode", 0)


def _in_mode(lw, mode, fn, *args):
    lw.set_option("mode", mode)
    try:
        return fn(*args)
    finally:
        lw.set_option("mode", 0)


def _lagrange_of(lw, mono, g2):
    s = _in_mode(lw, 1, lw.load_trusted_setup, b"".join(mono), b"".join(g2))
    try:
        return lagrange_from_settings(s)
    finally:
        s.free()


@pytest.fixture(scope="module")
def sec(lw):
    mono, g2 = golden_sections()
    lag = _lagrange_of(lw, mono, g2)
    return lag, g2, mono


def _file(data: bytes) -> str:
    f = tempfile.NamedTemporaryFile(suffix=".txt", delete=False)
    f.write(data)
    f.close()
    return f.name


def _load_file(lw, data: bytes, mode=0, precompute=0):
    path = _file(data)
    try:
        return _in_mode(lw, mode, lw.load_trusted_setup_file_ckzg, path, precompute)
    finally:
        os.unlink(path)


def _load_bytes(lw, lag, g2, mono, mode=0):
    return _in_mode(lw, mode, lw.load_trusted_setup_ckzg, b"".join(mono), b"".join(lag), b"".join(g2))


def test_lagrange_section_is_natural_order_over_tau(sec):
    from oracle.py import bls

    lag = sec[0]
    rng = random.Random(5)
    for k in [0, N - 1] + rng.sample(range(1, N - 1), 14):
        assert lag[k] == bls.g1_compress(bls.g1_mul(bls.G1, lagrange_scalar(k))), k


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_settings_equal_the_monomial_loader(lw, sec, mode):
    old = _in_mode(lw, mode, lw.load_trusted_setup_file, SETUP)
    try:
        want = (old.g1_values_bytes(), old.g2_values_bytes())
    finally:
        old.free()
    for s in [_load_file(lw, write_text(*sec), mode), _load_bytes(lw, *sec, mode=mode)]:
        try:
            assert (s.g1_values_bytes(), s.g2_values_bytes()) == want
        finally:
            s.free()


@pytest.fixture(scope="module")
def pair2(lw, sec):
    old = _in_mode(lw, 2, lw.load_trusted_setup_file, SETUP)
    new = _load_file(lw, write_text(*sec), 2)
    yield old, new
    old.free()
    new.free()


def test_mode2_outputs_equal(lw, pair2):
    old, new = pair2
    blobs = [lw.synth_blob_host(k) for k in range(8)]
    edge = [bytes(4096 * 32), (R - 1).to_bytes(32, "big") * 4096, R.to_bytes(32, "big") + bytes(4096 * 32 - 32)]
    all_blobs = b"".join(blobs + edge)
    a = lw.commit_and_prove_batch(all_blobs, len(blobs) + len(edge), old)
    b = lw.commit_and_prove_batch(all_blobs, len(blobs) + len(edge), new)
    assert a == b
    assert a[2][:10] == [0] * 10 and a[2][10] == lw.C_KZG_BADARGS
    coms, proofs = a[0][:8], a[1][:8]
    z = (123456789).to_bytes(32, "big")
    assert lw.compute_kzg_proof(blobs[3], z, old) == lw.compute_kzg_proof(blobs[3], z, new)
    for s in (old, new):
        assert lw.verify_blob_kzg_proof_batch(blobs, coms, proofs, s) is True
        bad = list(proofs)
        bad[2], bad[5] = bad[5], bad[2]
        assert lw.verify_blob_kzg_proof_batch(blobs, coms, bad, s) is False


def test_mode2_cells_equal_and_match_the_kats(lw, pair2):
    old, new = pair2
    kats = [e for e in json.load(open(os.path.join(GOLDEN, "cell_kats.json"))) if e["mode"] == 2]
    for e in kats:
        blob = make_blob(e["seed"], 2)
        cs, ps = lw.compute_cells_and_kzg_proofs(blob, new)
        assert (cs, ps) == lw.compute_cells_and_kzg_proofs(blob, old)
        assert hashlib.sha256(b"".join(cs)).hexdigest() == e["cells_sha256"]
        assert [ps[i].hex() for i in e["proof_cells"]] == e["proofs"]
        c = lw.blob_to_kzg_commitment(blob, new)
        assert c.hex() == e["commitment"]
        idx = [0, 5, 64, 127]
        for s in (old, new):
            assert lw.verify_cell_kzg_proof_batch([c] * 4, idx, [cs[i] for i in idx], [ps[i] for i in idx], s) is True
            assert lw.verify_cell_kzg_proof_batch([c] * 4, idx, [cs[i] for i in idx], [ps[5], ps[0], ps[64], ps[127]], s) is False
        keep = list(range(0, 128, 2))
        rec = lw.recover_cells_and_kzg_proofs(keep, [cs[i] for i in keep], new)
        assert rec == (cs, ps) == lw.recover_cells_and_kzg_proofs(keep, [cs[i] for i in keep], old)


def test_whitespace_variants_load_the_same(lw, sec):
    want = None
    for nl, fin in [("\n", True), ("\r\n", True), ("\r\n", False), ("\n", False)]:
        s = _load_file(lw, write_text(*sec, newline=nl, final_newline=fin))
        try:
            got = (s.g1_values_bytes(), s.g2_values_bytes())
        finally:
            s.free()
        want = want or got
        assert got == want, (nl, fin)
    # spaces between byte pairs and trailing content after the last point
    lag, g2, mono = sec
    spaced = write_text(lag, g2, mono).replace(mono[0].hex().encode(), b" ".join(mono[0][i: i + 1].hex().encode() for i in range(48)), 1)
    s = _load_file(lw, spaced + b"\ntrailing content is ignored\n")
    try:
        assert (s.g1_values_bytes(), s.g2_values_bytes()) == want
    finally:
        s.free()


def _g1(p):
    from oracle.py import bls

    return bls.g1_decompress(p)


def _g1c(p):
    from oracle.py import bls

    return bls.g1_compress(p)


def _rejections(lw, sec):
    from oracle.py import bls

    lag, g2, mono = sec
    swap = list(lag)
    swap[10], swap[11] = swap[11], swap[10]
    mono2 = list(mono)
    mono2[N - 1] = _g1c(bls.g1_add(_g1(mono[N - 1]), _g1(mono[N - 1])))
    g2_64 = list(g2)
    g2_64[64] = g2[63]
    g2_7 = list(g2)
    q7 = bls.g2_decompress(g2[7])
    g2_7[7] = bls.g2_compress(bls.g2_add(q7, q7))
    dbl = lambda pts: [_g1c(bls.g1_add(_g1(p), _g1(p))) for p in pts]  # noqa: E731
    g2_forged = list(g2)
    g2_forged[9] = forged_g2_outside_subgroup()
    x_big = list(lag)
    x_big[5] = bytes([0x80 | (bls.P >> 376)]) + (bls.P % (1 << 376)).to_bytes(47, "big")
    return {
        "two Lagrange points swapped": (swap, g2, mono, "Lagrange form"),
        "Lagrange section bit-reversed": ([lag[bitrev12(k)] for k in range(N)], g2, mono, "Lagrange form"),
        "monomial section as the Lagrange section": (mono, g2, mono, "Lagrange form"),
        "M_4095 doubled, Lagrange re-derived": (_lagrange_of(lw, mono2, g2), g2, mono2, "powers-of-tau chain"),
        "Q_64 = Q_63": (lag, g2_64, mono, "G2 point 64 does not continue"),
        "Q_7 doubled": (lag, g2_7, mono, "G2 point 7 does not continue"),
        "every G1 point doubled": (dbl(lag), g2, dbl(mono), "not the generator"),
        "G2 point outside G2": (lag, g2_forged, mono, "G2 point 9 is not in G2"),
        "G1 x >= p": (x_big, g2, mono, "Lagrange G1 point 5 is not a valid"),
    }


def test_inconsistent_setups_are_badargs(lw, sec):
    for name, (lag, g2, mono, why) in _rejections(lw, sec).items():
        for load in (lambda: _load_file(lw, write_text(lag, g2, mono), 2), lambda: _load_bytes(lw, lag, g2, mono, 2)):
            with pytest.raises(lw.KzgError) as ei:
                load()
            assert ei.value.code == lw.C_KZG_BADARGS, name
            assert why in lw.last_error(), (name, lw.last_error())


def test_malformed_input_is_badargs_and_out_untouched(lw, sec):
    lag, g2, mono = sec
    good = write_text(lag, g2, mono)
    bad_hex = bytearray(good)
    bad_hex[len(good) // 2] = ord("z")
    lib = lw.load_library()
    cases = [write_text(lag, g2, mono, header=(4096, 64)), good[: len(good) - 1000], bytes(bad_hex)]
    for data in cases:
        path = _file(data)
        try:
            libc = ctypes.CDLL(None)
            libc.fopen.restype = ctypes.c_void_p
            libc.fopen.argtypes = [ctypes.c_char_p, ctypes.c_char_p]
            libc.fclose.argtypes = [ctypes.c_void_p]
            fp = libc.fopen(path.encode(), b"rb")
            s = lw.Settings()
            ctypes.memset(s.ptr, 0x5A, ctypes.sizeof(s.c))
            assert lib.lwkzg_load_trusted_setup_file_ckzg(s.ptr, fp, 0) == lw.C_KZG_BADARGS
            libc.fclose(fp)
            assert ctypes.string_at(s.ptr, ctypes.sizeof(s.c)) == b"\x5a" * ctypes.sizeof(s.c)
        finally:
            os.unlink(path)
    m, l, q = b"".join(mono), b"".join(lag), b"".join(g2)
    s = lw.Settings()
    ctypes.memset(s.ptr, 0x5A, ctypes.sizeof(s.c))
    assert lib.lwkzg_load_trusted_setup_ckzg(s.ptr, m, len(m), l, len(l), q, len(q), 16) == lw.C_KZG_BADARGS
    assert lib.lwkzg_load_trusted_setup_ckzg(s.ptr, m, len(m) - 48, l, len(l), q, len(q), 0) == lw.C_KZG_BADARGS
    # a setup the device check rejects leaves *out untouched too
    swap = list(lag)
    swap[0], swap[1] = swap[1], swap[0]
    l2 = b"".join(swap)
    assert lib.lwkzg_load_trusted_setup_ckzg(s.ptr, m, len(m), l2, len(l2), q, len(q), 0) == lw.C_KZG_BADARGS
    assert ctypes.string_at(s.ptr, ctypes.sizeof(s.c)) == b"\x5a" * ctypes.sizeof(s.c)


def test_load_and_free_returns_device_memory(lw, sec):
    import torch

    data = write_text(*sec)
    _load_file(lw, data, 2).free()   # first-use allocations of the runtime and the library
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info()
    for _ in range(3):
        _load_file(lw, data, 2).free()
        try:
            _load_bytes(lw, list(reversed(sec[0])), sec[1], sec[2], 2)
        except lw.KzgError:
            pass
    torch.cuda.synchronize()
    free1, _ = torch.cuda.mem_get_info()
    assert abs(free1 - free0) <= 64 << 20, (free0, free1)


def test_table_shared_with_the_monomial_loader(lw, sec):
    lw.set_option("share_table", 1)
    try:
        old = _in_mode(lw, 2, lw.load_trusted_setup_file, SETUP)
        try:
            new = _load_file(lw, write_text(*sec), 2)
            try:
                assert lw.table_share(new) == 3
            finally:
                new.free()
        finally:
            old.free()
    finally:
        lw.set_option("share_table", 0)


def test_multi_device_equals_single_device(lw, pair2):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    _, new = pair2
    blobs = b"".join(lw.synth_blob_host(300 + k) for k in range(16))
    cblobs = b"".join(make_blob(40 + k, 2) for k in range(4))
    one = lw.commit_and_prove_batch(blobs, 16, new), lw.compute_cells_and_kzg_proofs_batch(cblobs, 4, new)
    lw.set_devices(list(range(torch.cuda.device_count())))
    try:
        many = lw.commit_and_prove_batch(blobs, 16, new), lw.compute_cells_and_kzg_proofs_batch(cblobs, 4, new)
    finally:
        lw.set_devices([])
    assert many == one
