"""c-kzg-4844 trusted-setup files for the tests: the golden tau = 1337 setup's sections, a writer and a reader of the
c-kzg text format (decimal counts 4096 / 65, then the Lagrange G1, G2 and monomial G1 points as hex, one per line)."""
import os

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TAU = 1337
N = 4096


def golden_sections():
    """(monomial G1, G2) compressed points of tests/golden/trusted_setup.txt (the reference's format)."""
    lines = open(os.path.join(GOLDEN, "trusted_setup.txt")).read().split("\n")
    n1, n2 = int(lines[0]), int(lines[1])
    mono = [bytes.fromhex(x) for x in lines[2: 2 + n1]]
    g2 = [bytes.fromhex(x) for x in lines[2 + n1: 2 + n1 + n2]]
    return mono, g2


def bitrev12(i: int) -> int:
    return int(format(i, "012b")[::-1], 2)


def lagrange_from_settings(s):
    """The natural-order Lagrange section from mode-1 or mode-2 settings: g1_values holds it bit-reversed, as
    blst_p1 (x, y, z; six u64 limbs each, most significant first)."""
    from oracle.py import bls

    raw = s.g1_values_bytes()

    def fp(off):
        limbs = [int.from_bytes(raw[off + 8 * k: off + 8 * k + 8], "little") for k in range(6)]
        v = 0
        for l in limbs:
            v = (v << 64) | l
        return v

    out = [None] * N
    for i in range(N):
        out[bitrev12(i)] = bls.g1_compress((fp(144 * i), fp(144 * i + 48)))
    return out


def write_text(lagrange, g2, mono, newline="\n", final_newline=True, header=(N, 65)) -> bytes:
    lines = ["%d" % header[0], "%d" % header[1]] + [p.hex() for p in list(lagrange) + list(g2) + list(mono)]
    text = newline.join(lines) + (newline if final_newline else "")
    return text.encode()


def read_text(data: bytes):
    """(lagrange, g2, monomial) of a c-kzg text file: whitespace-separated tokens."""
    tok = data.decode().split()
    assert tok[0] == "4096" and tok[1] == "65", tok[:2]
    hexs = "".join(tok[2:])
    pts = [bytes.fromhex(hexs[96 * i: 96 * i + 96]) for i in range(N)]
    off = 96 * N
    g2 = [bytes.fromhex(hexs[off + 192 * i: off + 192 * i + 192]) for i in range(65)]
    off += 192 * 65
    mono = [bytes.fromhex(hexs[off + 96 * i: off + 96 * i + 96]) for i in range(N)]
    return pts, g2, mono


def lagrange_scalar(k: int, tau: int = TAU) -> int:
    """l_k(tau) over the 4096th roots of unity in natural order: (w^k / n) (tau^n - 1) / (tau - w^k)."""
    from oracle.py import bls, kzg

    w_k = kzg.brp_domain()[bitrev12(k)]
    return w_k * (pow(tau, N, bls.R) - 1) * pow(N * (tau - w_k) % bls.R, -1, bls.R) % bls.R


def forged_g2_outside_subgroup():
    """A compressed point on the twist y^2 = x^3 + 4(1 + u) that is not in G2."""
    from oracle.py import bls

    for x0 in range(1, 100):
        x = (x0, 1)
        y = bls.fp2_sqrt(bls.fp2_add(bls.fp2_mul(bls.fp2_sqr(x), x), bls.B2))
        if y is None:
            continue
        pt = (x, y)
        assert bls.g2_on_curve(pt)
        if bls.g2_mul(pt, bls.R) is not None:
            return bls.g2_compress(pt)
    raise AssertionError("no point found")
