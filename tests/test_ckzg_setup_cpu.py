"""CPU tier: the c-kzg-4844 trusted-setup loaders reject bad arguments and malformed files with C_KZG_BADARGS before
they touch a device, and the tests' c-kzg file writer round-trips oracle-computed points."""
import ctypes
import os
import tempfile

import pytest

from tests._ckzg_setup import N, TAU, golden_sections, lagrange_scalar, read_text, write_text


@pytest.fixture(scope="module")
def lw():
    import lambdaworks_kzg_b200 as m

    m.load_library()
    return m


@pytest.fixture(scope="module")
def sections():
    mono, g2 = golden_sections()
    # any 4096 well-formed tokens do for the parser: the Lagrange section is only checked on the device
    return list(mono), g2, mono


def _no_gpu():
    try:
        import torch

        return not torch.cuda.is_available()
    except ImportError:
        return True


def _load_text(lw, data: bytes, precompute: int = 0):
    with tempfile.NamedTemporaryFile(suffix=".txt", delete=False) as f:
        f.write(data)
        path = f.name
    try:
        return lw.load_trusted_setup_file_ckzg(path, precompute)
    finally:
        os.unlink(path)


def _malformed(sections):
    lag, g2, mono = sections
    good = write_text(lag, g2, mono)
    bad_hex = bytearray(good)
    bad_hex[good.index(b"\n", 10) + 7] = ord("g")    # inside the first Lagrange point
    split_pair = good.replace(lag[3].hex().encode(), lag[3].hex()[:9].encode() + b" " + lag[3].hex()[9:].encode(), 1)
    return {
        "header 4096/64": write_text(lag, g2, mono, header=(4096, 64)),
        "header 4095/65": write_text(lag, g2, mono, header=(4095, 65)),
        "header not decimal": b"0x1000\n65\n" + good.split(b"\n", 2)[2],
        "truncated": good[: len(good) // 2],
        "one point short": write_text(lag, g2, mono[:-1]),
        "odd hex digit at the end": write_text(lag, g2, mono)[:-2],
        "non-hex character": bytes(bad_hex),
        "pair split by a space": split_pair,
        "empty": b"",
    }


@pytest.mark.parametrize("case", ["header 4096/64", "header 4095/65", "header not decimal", "truncated", "one point short",
                                  "odd hex digit at the end", "non-hex character", "pair split by a space", "empty"])
def test_malformed_file_is_badargs(lw, sections, case):
    with pytest.raises(lw.KzgError) as ei:
        _load_text(lw, _malformed(sections)[case])
    assert ei.value.code == lw.C_KZG_BADARGS, (case, lw.last_error())
    assert "c-kzg trusted setup" in lw.last_error()


def test_bad_arguments_are_badargs(lw, sections):
    lag, g2, mono = sections
    m, l, q = b"".join(mono), b"".join(lag), b"".join(g2)
    lib = lw.load_library()
    for args in [(m[:-48], l, q, 0), (m, l + bytes(48), q, 0), (m, l, q[:-1], 0), (m, l, q, 16), (m, l, q, 1 << 40)]:
        s = lw.Settings()
        ctypes.memset(s.ptr, 0x5A, ctypes.sizeof(s.c))
        rc = lib.lwkzg_load_trusted_setup_ckzg(s.ptr, args[0], len(args[0]), args[1], len(args[1]), args[2], len(args[2]), args[3])
        assert rc == lw.C_KZG_BADARGS, [len(a) if isinstance(a, bytes) else a for a in args]
        assert ctypes.string_at(s.ptr, ctypes.sizeof(s.c)) == b"\x5a" * ctypes.sizeof(s.c), "*out was written on failure"
    assert lib.lwkzg_load_trusted_setup_ckzg(None, m, len(m), l, len(l), q, len(q), 0) == lw.C_KZG_BADARGS
    s = lw.Settings()
    assert lib.lwkzg_load_trusted_setup_ckzg(s.ptr, None, len(m), l, len(l), q, len(q), 0) == lw.C_KZG_BADARGS
    assert lib.lwkzg_load_trusted_setup_file_ckzg(s.ptr, None, 0) == lw.C_KZG_BADARGS
    with pytest.raises(lw.KzgError) as ei:
        _load_text(lw, write_text(lag, g2, mono), precompute=16)
    assert ei.value.code == lw.C_KZG_BADARGS


@pytest.mark.skipif(not _no_gpu(), reason="a GPU is present")
def test_well_formed_file_needs_a_device(lw, sections):
    with pytest.raises(lw.KzgError) as ei:
        _load_text(lw, write_text(*sections, newline="\r\n", final_newline=False))
    assert ei.value.code == lw.C_KZG_ERROR


def test_writer_round_trips_oracle_points():
    from oracle.py import bls

    lag = [bls.g1_compress(bls.g1_mul(bls.G1, lagrange_scalar(k))) for k in (0, 1, N - 1)]
    mono = [bls.g1_compress(bls.g1_mul(bls.G1, pow(TAU, j, bls.R))) for j in range(3)]
    h = bls.g2_decompress(golden_sections()[1][0])   # the setup's G2 generator
    g2 = [bls.g2_compress(bls.g2_mul(h, pow(TAU, i, bls.R))) for i in range(2)]
    assert g2[1] == golden_sections()[1][1]
    lag_s = (lag * N)[:N]
    mono_s = (mono * N)[:N]
    g2_s = (g2 * 65)[:65]
    for nl, fin in [("\n", True), ("\r\n", True), ("\n", False), ("\r\n", False), (" ", False)]:
        assert read_text(write_text(lag_s, g2_s, mono_s, newline=nl, final_newline=fin)) == (lag_s, g2_s, mono_s)
    assert mono == golden_sections()[0][:3]
    assert sum(lagrange_scalar(k) for k in range(N)) % bls.R == 1   # the Lagrange basis sums to 1 at tau
