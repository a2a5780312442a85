"""The device math headers (mont/field/fpinv/g1/recode/fp2/sha256/lepoly/pairing) case by case against the Python
big-int oracle, on the GPU and under host emulation.

tests/device_math/harness.cu runs one case per thread.  The case tables are built so that the branches of each
operation are known per case (its class), and every table runs in four launch layouts with the same expected
values:
  mixed      lane i takes class i mod K: every warp executes every branch of the operation at once;
  uniform    cases sorted by class: whole warps agree;
  ragged     n not a multiple of 32 and a partial last block: the last warp is partial;
  divergent  only odd lanes call the operation, even lanes branch around it.
The emul backend runs the same tables on the host (one case after the other), so the tables and expected values
are checked without a GPU; warp-level behaviour (early-finishing lanes of the inversion, out-of-line calls,
funnel shifts, divergent branches) is only exercised by the device backend.

Field results are compared as exact limb values: a result must be the canonical representative (< modulus), not
merely congruent, because fp_eq / fp_is_zero compare limbs.  XYZZ results are checked without any device inversion:
ZZ^3 == ZZZ^2, affine = (X/ZZ, Y/ZZZ) in Python, infinity iff ZZ == 0.
"""
import functools
import hashlib
import random

import pytest

from oracle.py import bls
from tests._device_math import Harness, bytes_words, from_words, words, words_bytes

P, R = bls.P, bls.R
RP, RR = 1 << 384, 1 << 256
RP_INV, RR_INV = pow(RP, -1, P), pow(RR, -1, R)
X2 = bls.BLS_X ** 2

# operation ids of harness.cu
OP_FP_ARITH, OP_FR_ARITH, OP_FP_FROM_BE48, OP_FR_FROM_BE = 0, 1, 2, 3
OP_FP_INV_GCD, OP_FP_INV_FERMAT, OP_FR_INV, OP_FR_BATCH_INV, OP_FR_ZN_MINUS_ONE = 4, 5, 6, 7, 8
OP_XYZZ_MADD, OP_XYZZ_MADD_HOT, OP_XYZZ_MADD_NI, OP_XYZZ_MADD_RARE = 10, 11, 12, 13
OP_XYZZ_ADD, OP_XYZZ_ADD_NI, OP_XYZZ_DBL, OP_XYZZ_DBL_NI = 14, 15, 16, 17
OP_XYZZ_DBL_AFFINE, OP_G1A_DBL_NI, OP_XYZZ_TO_AFFINE, OP_XYZZ_EQ = 18, 19, 20, 21
OP_G1_MUL, OP_GLV_RECODE = 30, 31
OP_G1_COMPRESS, OP_G1_DECOMPRESS, OP_G1_DECOMPRESS_NOSUB, OP_G1_DECOMPRESS_STRICT = 40, 41, 42, 43
OP_G1_CHECKS, OP_G2_DECOMPRESS, OP_FP2_INV, OP_FP2_SQRT = 44, 45, 46, 47
OP_SHA256_ONESHOT, OP_SHA256_WARP, OP_PAIRING = 50, 51, 60

LAYOUTS = ["mixed", "uniform", "ragged", "divergent"]


@pytest.fixture(scope="module", params=["emul", pytest.param("device", marks=pytest.mark.gpu)])
def hx(request):
    return Harness(request.param)


def device_only(hx):
    if hx.backend != "device":
        pytest.skip("device-only piece of the headers (not compiled under host emulation)")


# ------------------------------------------------------------------ layouts
def round_robin(classes):
    """Case indices, lane i taking class i mod K while every class has cases left."""
    queues = [list(v) for v in classes.values()]
    order = []
    while any(queues):
        for q in queues:
            if q:
                order.append(q.pop(0))
    return order


def arrange(cls, layout):
    """cls: class of each case -> (case order, threads per block, odd_lanes_only)."""
    classes = {}
    for i, c in enumerate(cls):
        classes.setdefault(c, []).append(i)
    if layout == "uniform":
        return [i for c in classes for i in classes[c]], 32, False
    order = round_robin(classes)
    if layout == "mixed":
        return order, 64, False
    if layout == "ragged":
        extra = (5 - len(order)) % 32 or 32
        order = order + order[:extra]
        assert len(order) % 32 != 0
        return order, 96, False
    assert layout == "divergent"
    return order, 64, True


def run_layout(hx, op, records, cls, out_words, layout):
    """Runs the table in the given layout; results come back in case order.  A case that runs twice (the ragged
    layout repeats a few) must give the same words both times."""
    order, tpb, odd = arrange(cls, layout)
    outs = hx.run(op, [records[i] for i in order], out_words, tpb, odd)
    if outs is None:
        device_only(hx)
    res = [None] * len(records)
    for j, i in enumerate(order):
        assert res[i] is None or res[i] == outs[j], "case %d differs between two lanes" % i
        res[i] = outs[j]
    return res


def balanced(groups, per=None):
    """{class: [case, ...]} -> (cases, classes) with every class cycled to the same count."""
    per = per or max(len(v) for v in groups.values())
    cases, cls = [], []
    for c, v in groups.items():
        assert v, c
        for j in range(per):
            cases.append(v[j % len(v)])
            cls.append(c)
    return cases, cls


def canon(w, m):
    v = from_words(w)
    assert v < m, "non-canonical limbs: %#x >= modulus" % v
    return v


def mont_fp(v):
    return words(v * RP % P, 12)


def aff_words(pt):
    return words(0, 24) if pt is None else mont_fp(pt[0]) + mont_fp(pt[1])


def xyzz_words(pt, lam=1):
    """XYZZ (Montgomery) of an affine point scaled by lam: (x lam^2, y lam^3, lam^2, lam^3); infinity = zeros."""
    if pt is None:
        return words(0, 48)
    l2, l3 = lam * lam % P, lam * lam * lam % P
    return mont_fp(pt[0] * l2 % P) + mont_fp(pt[1] * l3 % P) + mont_fp(l2) + mont_fp(l3)


def xyzz_point(w):
    """G1Xyzz words -> affine point (or None), checking the invariants."""
    X, Y, ZZ, ZZZ = (canon(w[12 * i:12 * i + 12], P) * RP_INV % P for i in range(4))
    if ZZ == 0:
        return None
    assert pow(ZZ, 3, P) == pow(ZZZ, 2, P), "ZZ^3 != ZZZ^2"
    return (X * bls.fp_inv(ZZ) % P, Y * bls.fp_inv(ZZZ) % P)


def aff_point(w):
    x, y = canon(w[:12], P), canon(w[12:24], P)
    if x == 0 and y == 0:
        return None
    return (x * RP_INV % P, y * RP_INV % P)


# ------------------------------------------------------------------ Fp / Fr arithmetic
def _edges(m, nlimbs):
    half_bits = 32 * nlimbs // 2
    hi = (m >> half_bits) << half_bits
    R_ = (1 << (32 * nlimbs)) % m
    top = 1 << (m.bit_length() - 2)
    return sorted({0, 1, 2, m - 1, m - 2, (m - 1) // 2, (m + 1) // 2, top, top - 1,
                   (1 << half_bits) - 1, hi - 1, R_, R_ * R_ % m})


@functools.lru_cache(maxsize=None)
def arith_table(m, nlimbs):
    rnd = random.Random(m & 0xFFFF)
    RM = 1 << (32 * nlimbs)
    E = _edges(m, nlimbs)

    def ra():
        return rnd.randrange(2, m - 1)

    g = {"edge": [(a, b) for a in E for b in E]}
    n = len(g["edge"])
    g["sum=m-1"] = [(a, m - 1 - a) for a in (ra() for _ in range(n))]
    g["sum=m"] = [(a, m - a) for a in (ra() for _ in range(n))] + [(1, m - 1), (m - 1, 1), ((m - 1) // 2, (m + 1) // 2)]
    g["sum=m+1"] = [(a, m + 1 - a) for a in (ra() for _ in range(n))]
    g["sum=2m-2"] = [(m - 1, m - 1)]
    g["diff=0"] = [(a, a) for a in E + [ra() for _ in range(n)]]
    g["diff=-1"] = [(a, a + 1) for a in [ra() for _ in range(n)] + [0, m - 2]]
    g["diff=1-m"] = [(0, m - 1)]
    inv = {a: pow(a, -1, m) for a in [ra() for _ in range(n)] + [1, 2, m - 1]}
    g["prod=0"] = [(a, 0) for a in inv] + [(0, a) for a in inv]
    g["prod=1"] = [(a, ai * RM % m) for a, ai in inv.items()]
    g["prod=m-1"] = [(a, (m - 1) * ai * RM % m) for a, ai in inv.items()]
    g["random"] = [(ra(), ra()) for _ in range(n)]
    cases, cls = balanced(g)
    for (a, b), c in zip(cases, cls):
        assert 0 <= a < m and 0 <= b < m
        if c.startswith("sum="):
            assert a + b == {"sum=m-1": m - 1, "sum=m": m, "sum=m+1": m + 1, "sum=2m-2": 2 * m - 2}[c]
    return cases, cls


def arith_expect(m, nlimbs, a, b, with_nv):
    inv = pow(1 << (32 * nlimbs), -1, m)
    RM = (1 << (32 * nlimbs)) % m
    mul, sqr = a * b * inv % m, a * a * inv % m
    out = [(a + b) % m, (a - b) % m, (-a) % m, 2 * a % m, mul]
    out += [mul, sqr, sqr] if with_nv else [sqr]
    return out + [a * RM % m, a * inv % m]


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("field", ["fp", "fr"])
def test_field_arith(hx, field, layout):
    m, nl, op, with_nv, names = ((P, 12, OP_FP_ARITH, True, "add sub neg dbl mul mul_nv sqr sqr_nv to_mont from_mont")
                                 if field == "fp" else
                                 (R, 8, OP_FR_ARITH, False, "add sub neg dbl mul sqr to_mont from_mont"))
    names = names.split()
    cases, cls = arith_table(m, nl)
    res = run_layout(hx, op, [words(a, nl) + words(b, nl) for a, b in cases], cls, nl * len(names), layout)
    for (a, b), c, out in zip(cases, cls, res):
        want = arith_expect(m, nl, a, b, with_nv)
        for k, name in enumerate(names):
            got = from_words(out[nl * k:nl * (k + 1)])
            assert got == want[k], "%s_%s(%#x, %#x) [%s]: got %#x (%s)" % (
                field, name, a, b, c, got, "non-canonical" if got % m == want[k] else "wrong value")


@pytest.mark.parametrize("layout", LAYOUTS)
def test_byte_decoders(hx, layout):
    """fp_from_be48 reduces x < 2^381 (including p <= x < 2p) into Montgomery form; fr_canon_from_be32 and the
    byte-permute path fr_canon_from_be_words reduce any 256-bit value (up to two subtractions)."""
    rnd = random.Random(21)
    xs = {"x<p": [0, 1, P - 1, P - 2] + [rnd.randrange(P) for _ in range(12)],
          "x>=p": [P, P + 1, P + 2, (1 << 381) - 1]
          + [rnd.randrange(P, 1 << 381) for _ in range(12)]}
    cases, cls = balanced(xs)
    res = run_layout(hx, OP_FP_FROM_BE48, [bytes_words(x.to_bytes(48, "big")) for x in cases], cls, 12, layout)
    for x, out in zip(cases, res):
        assert from_words(out) == x % P * RP % P, hex(x)
    vs = {"v<r": [0, 1, R - 1] + [rnd.randrange(R) for _ in range(8)],
          "r<=v<2r": [R, R + 1, 2 * R - 1] + [rnd.randrange(R, 2 * R) for _ in range(8)],
          "v>=2r": [2 * R, 2 * R + 1, (1 << 256) - 1] + [rnd.randrange(2 * R, 1 << 256) for _ in range(8)]}
    cases, cls = balanced(vs)
    res = run_layout(hx, OP_FR_FROM_BE, [bytes_words(v.to_bytes(32, "big")) for v in cases], cls, 16, layout)
    for v, out in zip(cases, res):
        assert from_words(out[:8]) == v % R, ("be32", hex(v))
        assert from_words(out[8:]) == v % R, ("be_words", hex(v))


# ------------------------------------------------------------------ inversion
def gcd_rounds(a):
    """(rounds until a == 0, rounds until b == 1) of fpinv.cuh's approximate binary GCD on input a: the same 62-bit
    approximations, 30 divsteps per round, exact matrix application.  The loop runs until a == 0 in every lane of
    the warp (the maximum over its lanes); the value is fixed once b == 1 -- the rounds after that only shift a down
    and divide the cofactor by 4, which the final 4^rounds scale undoes."""
    M32, M64 = (1 << 32) - 1, (1 << 64) - 1

    def s32(x):
        return x - (1 << 32) if x >> 31 else x

    b, rounds, settled = P, 0, 0
    while a:
        al = [(a >> (32 * i)) & M32 for i in range(12)]
        bl = [(b >> (32 * i)) & M32 for i in range(12)]
        top = next((i for i in range(11, 0, -1) if al[i] | bl[i]), None)
        c = 32 if top is None else 32 - (al[top] | bl[top]).bit_length()
        if top is None or (top == 1 and c >= 3):
            abar, bbar = a & M64, b & M64
        else:
            def approx(lim):
                hi = ((lim[top] << c) | (lim[top - 1] >> (32 - c))) & M32 if c else lim[top]
                return (hi << 30) | (lim[0] & 0x3FFFFFFF)
            abar, bbar = approx(al), approx(bl)
        f0, g0, f1, g1 = 1, 0, 0, 1
        for _ in range(30):
            if abar & 1:
                if abar < bbar:
                    abar, bbar, f0, f1, g0, g1 = bbar, abar, f1, f0, g1, g0
                abar -= bbar
                f0, g0 = (f0 - f1) & M32, (g0 - g1) & M32
            abar >>= 1
            f1, g1 = (f1 << 1) & M32, (g1 << 1) & M32
        na, nb = a * s32(f0) + b * s32(g0), a * s32(f1) + b * s32(g1)
        assert na % (1 << 30) == 0 and nb % (1 << 30) == 0
        a, b = abs(na) >> 30, abs(nb) >> 30
        rounds += 1
        if b == 1 and not settled:
            settled = rounds
    return rounds, settled


# The highest counts the tables reach (fpinv.cuh: MAX_ROUNDS = 30, "observed maximum 26"): 26 rounds until a == 0 for
# 2^k and p - 2^k, k in [370, 380]; 20 rounds until b == 1, the most a hill-climbing search over the model found (from
# p - 2^k + 1 and random starts) -- a loop cut after 20 or more rounds gives the same value on every input known here.
MAX_ROUNDS_REACHED = 26
MAX_SETTLE_REACHED = 20
SETTLE_20 = [P - (1 << 310) + 1, P - (1 << 356) + 1, P - (1 << 372) + 1,
             0x1a0111ea3917f48a0ad9e7b7c34a06e720233a84b38533b36510caa1d6b0fe241a2bfe7eb1537fbfb1faffffffffeaac,
             0xa0113ca355ff6aa5ad985bb2b6bac5725776b84f28512af077292e0f6b0f224dea3ffffb153ffffb9feffffffffaaac,
             0x1a01112a317ff6d24a992ea6434badf735734b89f38f3cb76710c2a174b026241eabfffeb151f7bfb9fefffefffeaaac]


@functools.lru_cache(maxsize=None)
def fp_inv_table():
    rnd = random.Random(31)
    vals = [1, 2, 3, P - 1, P - 2, (P - 1) // 2, RP % P] + [1 << k for k in range(0, 381, 19)]
    vals += [(1 << k) - 1 for k in range(2, 381, 23)] + [P - (1 << k) for k in range(1, 380, 29)]
    vals += [rnd.randrange(1, P) for _ in range(40)]
    vals += [1 << k for k in range(340, 381)] + [P - (1 << k) for k in range(340, 381)]   # the 25- and 26-round inputs
    groups = {"zero": [0], "b=1 after 20 rounds": SETTLE_20}
    for v in vals:
        r = gcd_rounds(v)[0]
        groups.setdefault("rounds<=19" if r <= 19 else "rounds 20-24" if r <= 24 else "rounds=%d" % r, []).append(v)
    assert max(gcd_rounds(v)[0] for v in groups["rounds=26"]) == MAX_ROUNDS_REACHED
    assert all(gcd_rounds(v)[1] == MAX_SETTLE_REACHED for v in SETTLE_20)
    return balanced(groups)


def fp_inv_expect(a):
    return 0 if a == 0 else pow(a * RP_INV % P, -1, P) * RP % P


@pytest.mark.parametrize("layout", LAYOUTS)
def test_fp_inversions(hx, layout):
    """fp_inv_gcd (what every caller uses) and fp_inv_fermat, Montgomery in and out, 0 -> 0.  In the mixed layout
    every warp holds a zero lane, lanes done after ~13 rounds, lanes that need 25 and 26 rounds and lanes whose b
    reaches 1 only in round 20, so lanes that finished keep running rounds until the whole warp is done (their
    cofactor keeps being divided by 4, which the final 4^rounds scale must match)."""
    cases, cls = fp_inv_table()
    recs = [words(a, 12) for a in cases]
    if layout == "mixed":
        order, _, _ = arrange(cls, layout)
        warps = [order[i:i + 32] for i in range(0, len(order) - 31, 32)]
        assert warps and all(max(gcd_rounds(cases[i])[0] for i in w) == MAX_ROUNDS_REACHED and
                             max(gcd_rounds(cases[i])[1] for i in w) == MAX_SETTLE_REACHED and
                             any(cases[i] == 0 for i in w) for w in warps)
    for op in (OP_FP_INV_GCD, OP_FP_INV_FERMAT):
        res = run_layout(hx, op, recs, cls, 12, layout)
        for a, c, out in zip(cases, cls, res):
            assert from_words(out) == fp_inv_expect(a), (op, c, hex(a))


def test_fp_inversion_warps(hx):
    """Whole warps composed on purpose: 32 equal values; one zero lane among 31 non-zero ones; one 26-round lane
    among 31 random ones (at lane 0, 17 and 31); a warp of 26-round lanes only.  Then the same warps with only the
    odd lanes calling the inversion."""
    rnd = random.Random(32)
    slow = [1 << k for k in range(370, 381)] + [P - (1 << k) for k in range(370, 381)]
    warps = [[rnd.randrange(1, P)] * 32, [P - 1] * 32, [0] * 32]
    w = [rnd.randrange(1, P) for _ in range(32)]
    w[13] = 0
    warps.append(w)
    for lane in (0, 17, 31):
        w = [rnd.randrange(1, P) for _ in range(32)]
        w[lane] = slow[lane % len(slow)]
        warps.append(w)
    warps.append([slow[i % len(slow)] for i in range(32)])
    cases = [v for w in warps for v in w]
    assert max(gcd_rounds(v)[0] for v in cases) == MAX_ROUNDS_REACHED
    for odd in (False, True):
        outs = hx.run(OP_FP_INV_GCD, [words(a, 12) for a in cases], 12, 32, odd)
        for i, (a, out) in enumerate(zip(cases, outs)):
            assert from_words(out) == fp_inv_expect(a), (i // 32, i % 32, hex(a), odd)


@pytest.mark.parametrize("layout", LAYOUTS)
def test_fr_inversion(hx, layout):
    rnd = random.Random(33)
    g = {"zero": [0], "edge": [1, 2, R - 1, R - 2, RR % R] + [1 << k for k in range(0, 255, 31)] + [(1 << k) - 1 for k in range(2, 255, 37)],
         "random": [rnd.randrange(1, R) for _ in range(16)]}
    cases, cls = balanced(g)
    res = run_layout(hx, OP_FR_INV, [words(a, 8) for a in cases], cls, 8, layout)
    for a, out in zip(cases, res):
        assert from_words(out) == (0 if a == 0 else pow(a * RR_INV % R, -1, R) * RR % R), hex(a)


@pytest.mark.parametrize("layout", LAYOUTS)
def test_fr_batch_inversion_and_vanishing(hx, layout):
    """fr_batch_inv_group (Montgomery's trick over a group of up to 32; zero entries give 0 and stay out of the
    running product) and fr_zn_minus_one (z^4096 - 1: exactly 0 on the domain)."""
    rnd = random.Random(34)
    B = 32

    def group(cnt, zeros):
        d = [0 if k in zeros else rnd.randrange(1, R) for k in range(cnt)]
        return [cnt] + sum((words(v, 8) for v in d + [0] * (B - cnt)), [])

    g = {"no zero": [group(32, ()), group(1, ()), group(7, ())],
         "zero first": [group(32, (0,)), group(5, (0,))],
         "zero last": [group(32, (31,)), group(9, (8,))],
         "zeros inside": [group(32, (3, 4, 17)), group(32, tuple(range(1, 32, 2)))],
         "all zero": [group(32, tuple(range(32))), group(1, (0,))]}
    cases, cls = balanced(g)
    res = run_layout(hx, OP_FR_BATCH_INV, cases, cls, 8 * B, layout)
    for rec, c, out in zip(cases, cls, res):
        for k in range(B):
            d = from_words(rec[1 + 8 * k:9 + 8 * k])
            want = 0 if d == 0 or k >= rec[0] else pow(d * RR_INV % R, -1, R) * RR % R
            assert from_words(out[8 * k:8 * k + 8]) == want, (c, rec[0], k)
    w = pow(7, (R - 1) // 4096, R)
    assert pow(w, 2048, R) != 1
    g = {"domain": [pow(w, j, R) for j in (0, 1, 2, 1024, 2048, 4095, 3000)],
         "off": [0, 2, R - 2, pow(7, (R - 1) // 8192, R)] + [rnd.randrange(R) for _ in range(3)]}
    cases, cls = balanced(g)
    res = run_layout(hx, OP_FR_ZN_MINUS_ONE, [words(z * RR % R, 8) for z in cases], cls, 8, layout)
    for z, c, out in zip(cases, cls, res):
        want = (pow(z, 4096, R) - 1) % R
        assert (want == 0) == (c == "domain")
        assert from_words(out) == want * RR % R, (c, hex(z))


# ------------------------------------------------------------------ G1 group law
G1_CLASSES = ["inf+P", "P+inf", "inf+inf", "P+P", "P-P", "P+Q", "P+2P"]


@functools.lru_cache(maxsize=None)
def g1_table():
    """Cases (A, B, lamA, lamB): accumulator A as XYZZ scaled by lamA (1: ZZ = ZZZ = 1), the other operand B as
    affine and as XYZZ scaled by lamB; 7 operand classes x {unscaled, scaled} = 14 classes."""
    rnd = random.Random(41)
    g = {}
    for i in range(6):
        p = bls.g1_mul(bls.G1, rnd.randrange(1, R))
        q = bls.g1_mul(bls.G1, rnd.randrange(1, R))
        pairs = {"inf+P": (None, p), "P+inf": (p, None), "inf+inf": (None, None), "P+P": (p, p),
                 "P-P": (p, bls.g1_neg(p)), "P+Q": (p, q), "P+2P": (p, bls.g1_add(p, p))}
        for scaled in (False, True):
            for c in G1_CLASSES:
                a, b = pairs[c]
                la, lb = (rnd.randrange(2, P), rnd.randrange(2, P)) if scaled else (1, 1)
                g.setdefault((c, scaled), []).append((a, b, la, lb))
    return balanced(g)


G1_OPS = {  # op: (expected point from A, B; output words, output kind)
    OP_XYZZ_MADD: (lambda a, b: bls.g1_add(a, b), 48, "xyzz"),
    OP_XYZZ_MADD_HOT: (lambda a, b: bls.g1_add(a, b), 48, "xyzz"),
    OP_XYZZ_MADD_NI: (lambda a, b: bls.g1_add(a, b), 48, "xyzz"),
    OP_XYZZ_MADD_RARE: (lambda a, b: bls.g1_add(a, b), 48, "xyzz"),
    OP_XYZZ_ADD: (lambda a, b: bls.g1_add(a, b), 48, "xyzz"),
    OP_XYZZ_ADD_NI: (lambda a, b: bls.g1_add(a, b), 48, "xyzz"),
    OP_XYZZ_DBL: (lambda a, b: bls.g1_add(a, a), 48, "xyzz"),
    OP_XYZZ_DBL_NI: (lambda a, b: bls.g1_add(a, a), 48, "xyzz"),
    OP_XYZZ_DBL_AFFINE: (lambda a, b: bls.g1_add(b, b), 48, "xyzz"),
    OP_G1A_DBL_NI: (lambda a, b: bls.g1_add(b, b), 24, "affine"),
    OP_XYZZ_TO_AFFINE: (lambda a, b: a, 24, "affine"),
    OP_XYZZ_EQ: (lambda a, b: a == b, 1, "flag"),
}
G1_OP_NAMES = {OP_XYZZ_MADD: "xyzz_madd", OP_XYZZ_MADD_HOT: "xyzz_madd_hot", OP_XYZZ_MADD_NI: "xyzz_madd_ni",
               OP_XYZZ_MADD_RARE: "xyzz_madd_rare", OP_XYZZ_ADD: "xyzz_add", OP_XYZZ_ADD_NI: "xyzz_add_ni",
               OP_XYZZ_DBL: "xyzz_dbl", OP_XYZZ_DBL_NI: "xyzz_dbl_ni", OP_XYZZ_DBL_AFFINE: "xyzz_dbl_affine",
               OP_G1A_DBL_NI: "g1a_dbl_ni", OP_XYZZ_TO_AFFINE: "xyzz_to_affine", OP_XYZZ_EQ: "xyzz_eq"}


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("op", list(G1_OPS), ids=[G1_OP_NAMES[o] for o in G1_OPS])
def test_g1_group_law(hx, op, layout):
    cases, cls = g1_table()
    if layout == "mixed":   # every warp of the mixed layout runs all 14 classes at once
        order, _, _ = arrange(cls, layout)
        warps = [order[i:i + 32] for i in range(0, len(order) - 31, 32)]
        assert warps and all({cls[i] for i in w} == set(cls) for w in warps)
    recs = [xyzz_words(a, la) + aff_words(b) + xyzz_words(b, lb) for a, b, la, lb in cases]
    fn, nout, kind = G1_OPS[op]
    res = run_layout(hx, op, recs, cls, nout, layout)
    for (a, b, la, lb), c, out in zip(cases, cls, res):
        want = fn(a, b)
        if kind == "xyzz":
            got = xyzz_point(out)
        elif kind == "affine":
            got = aff_point(out)
        else:
            got = bool(out[0])
        assert got == want, (G1_OP_NAMES[op], c)


# ------------------------------------------------------------------ scalars and recoding
GLV_EDGE = [0, 1, 2, R - 1, R - 2, (R - 1) // 2, (1 << 254) - 1, X2 - 1, X2, X2 + 1, (X2 - 2) * X2 + X2 - 1,
            5 * X2 - 1, 5 * X2, ((1 << 128) - 1) % R, (X2 - 1) * X2, 1 << 128, 2 * X2]


@pytest.mark.parametrize("layout", LAYOUTS)
def test_g1_scalar_mul(hx, layout):
    """g1_mul_scalar and g1_mul_scalar_glv (which returns early for an infinite base, after the split) with the
    infinite base inside warps of finite ones."""
    rnd = random.Random(51)
    pts = [bls.G1] + [bls.g1_mul(bls.G1, rnd.randrange(1, R)) for _ in range(3)]
    g = {"inf base": [(None, k) for k in GLV_EDGE[:6] + [rnd.randrange(R)]],
         "edge k": [(pts[i % 4], k) for i, k in enumerate(GLV_EDGE)],
         "random k": [(pts[i % 4], rnd.randrange(R)) for i in range(8)]}
    cases, cls = balanced(g, per=12)
    res = run_layout(hx, OP_G1_MUL, [aff_words(p) + words(k, 8) for p, k in cases], cls, 96, layout)
    want = {(p, k): bls.g1_mul(p, k) if p is not None else None for p, k in set(cases)}
    for (p, k), c, out in zip(cases, cls, res):
        assert xyzz_point(out[:48]) == want[(p, k)], ("g1_mul_scalar", c, hex(k))
        assert xyzz_point(out[48:]) == want[(p, k)], ("g1_mul_scalar_glv", c, hex(k))


@pytest.mark.parametrize("layout", LAYOUTS)
def test_glv_split_and_digits(hx, layout):
    """glv_split (bit-serial) and glv_split_barrett give k = m + q x^2; the signed digits of both halves for
    c in {8, 13, 16} add up to the half, lower windows in (-2^(c-1), 2^(c-1)], the top one in [0, top count]."""
    rnd = random.Random(52)
    g = {c: [(k, c) for k in GLV_EDGE + [rnd.randrange(R) for _ in range(40)]] for c in (8, 13, 16)}
    cases, cls = balanced(g)
    res = run_layout(hx, OP_GLV_RECODE, [words(0, 24) + words(k, 8) + [c] for k, c in cases], cls, 48, layout)
    for (k, c), out in zip(cases, res):
        qm = divmod(k, X2)
        assert (from_words(out[0:4]), from_words(out[4:8])) == qm, ("glv_split", hex(k))
        assert (from_words(out[8:12]), from_words(out[12:16])) == qm, ("glv_split_barrett", hex(k))
        W = -(-128 // c)
        top = ((X2 - 1) >> (c * (W - 1))) + 1
        for h, v in ((0, qm[1]), (1, qm[0])):
            d = [x - (1 << 32) if x >> 31 else x for x in out[16 + 16 * h:16 + 16 * h + W]]
            assert sum(x << (c * j) for j, x in enumerate(d)) == v, ("digits", c, h, hex(k))
            assert all(-(1 << (c - 1)) < x <= (1 << (c - 1)) for x in d[:-1]), ("digit range", c, h, hex(k))
            assert 0 <= d[-1] <= top, ("top digit", c, h, hex(k))


# ------------------------------------------------------------------ codecs
def _not_in_subgroup(rnd):
    while True:
        x = rnd.randrange(P)
        y = bls.fp_sqrt((x ** 3 + 4) % P)
        if y is not None and not bls.g1_in_subgroup((x, y)):
            return (x, y)


def _decompress_nosub(b):
    if not b[0] & 0x80:
        return "reject"
    if b[0] & 0x40:
        return None
    x = int.from_bytes(bytes([b[0] & 0x1F]) + b[1:], "big") % P
    y = bls.fp_sqrt((x ** 3 + 4) % P)
    if y is None:
        return "reject"
    lo, hi = (y, P - y) if y < P - y else (P - y, y)
    return (x, hi if b[0] & 0x20 else lo)


def _decompress_ref(b, strict):
    try:
        return bls.g1_decompress(b, strict=strict)
    except bls.PointError:
        return "reject"


@functools.lru_cache(maxsize=None)
def g1_codec_table():
    rnd = random.Random(61)
    pts = [bls.G1, bls.g1_neg(bls.G1)] + [bls.g1_mul(bls.G1, rnd.randrange(1, R)) for _ in range(4)]
    comp = [bls.g1_compress(p) for p in pts]
    x_off = [x for x in range(2, 200) if bls.fp_sqrt((x ** 3 + 4) % P) is None][:4]
    big = []
    for p in pts + [bls.g1_mul(bls.G1, rnd.randrange(1, R)) for _ in range(12)]:
        if p[0] + P < 1 << 381:
            b = bytearray((p[0] + P).to_bytes(48, "big"))
            b[0] |= 0x80 | (0x20 if (P - p[1]) % P < p[1] else 0)
            big.append(bytes(b))
    assert big
    ns = [_not_in_subgroup(rnd) for _ in range(3)]
    g = {"valid": comp,
         "sign flip": [bytes([c[0] ^ 0x20]) + c[1:] for c in comp],
         "infinity": [bytes([0xC0]) + bytes(47)],
         "infinity, junk": [bytes([0xE0]) + bytes(47), bytes([0xC0]) + b"\x01" + bytes(46), bytes([0xC0]) + bytes(46) + b"\x01"],
         "no flag": [bytes(48), bytes([0x40]) + bytes(47), bytes([comp[2][0] & 0x7F]) + comp[2][1:]],
         "x >= p": big,
         "x not on curve": [bytes([0x80]) + x.to_bytes(47, "big") for x in x_off],
         "not in subgroup": [bls.g1_compress(p) for p in ns]}
    return balanced(g)


@pytest.mark.parametrize("layout", LAYOUTS)
def test_g1_decompress(hx, layout):
    """Lax decoder with and without the subgroup check, and the strict decoder; accepted and rejected encodings
    share every warp of the mixed layout."""
    cases, cls = g1_codec_table()
    recs = [bytes_words(b) for b in cases]
    for op, ref in ((OP_G1_DECOMPRESS, lambda b: _decompress_ref(b, False)),
                    (OP_G1_DECOMPRESS_NOSUB, _decompress_nosub),
                    (OP_G1_DECOMPRESS_STRICT, lambda b: _decompress_ref(b, True))):
        res = run_layout(hx, op, recs, cls, 25, layout)
        for b, c, out in zip(cases, cls, res):
            want = ref(b)
            assert out[0] == (0 if want == "reject" else 1), (op, c, b.hex())
            assert aff_point(out[1:]) == (None if want == "reject" else want), (op, c, b.hex())
    strict_x_big = [cases[i] for i in range(len(cases)) if cls[i] == "x >= p"]
    assert all(_decompress_ref(b, False) != "reject" and _decompress_ref(b, True) == "reject" for b in strict_x_big)


@pytest.mark.parametrize("layout", LAYOUTS)
def test_g1_compress_and_checks(hx, layout):
    rnd = random.Random(62)
    good = [None, bls.G1, bls.g1_neg(bls.G1)] + [bls.g1_mul(bls.G1, rnd.randrange(1, R)) for _ in range(3)]
    cases, cls = balanced({"inf": [None], "point": good[1:]})
    res = run_layout(hx, OP_G1_COMPRESS, [aff_words(p) for p in cases], cls, 12, layout)
    for p, out in zip(cases, res):
        assert words_bytes(out) == bls.g1_compress(p)
    ns = _not_in_subgroup(rnd)
    tors = bls.g1_mul(ns, R)
    g = {"in subgroup": [(p, True, True) for p in good],
         "not in subgroup": [(ns, True, False), (tors, True, False), ((0, 2), True, False)],
         "off curve": [((bls.G1[0], (bls.G1[1] + 1) % P), False, None), ((1, 1), False, None)]}
    cases, cls = balanced(g)
    res = run_layout(hx, OP_G1_CHECKS, [aff_words(p) for p, _, _ in cases], cls, 2, layout)
    for (p, on, sub), c, out in zip(cases, cls, res):
        assert out[0] == (1 if on and p is not None else 0), ("on_curve", c)
        if sub is not None:
            assert out[1] == (1 if sub else 0), ("in_subgroup", c)


def _fp2_words(a):
    return mont_fp(a[0]) + mont_fp(a[1])


def _fp2_from(w):
    return (canon(w[:12], P) * RP_INV % P, canon(w[12:24], P) * RP_INV % P)


@pytest.mark.parametrize("layout", LAYOUTS)
def test_g2_decompress_and_fp2(hx, layout, py_setup):
    rnd = random.Random(63)
    raws = [bls.g2_compress(q) for q in py_setup.g2[:4]]
    x_off = next(x for x in range(1, 200) if bls.fp2_sqrt(bls.fp2_add(bls.fp2_mul(bls.fp2_sqr((x, 1)), (x, 1)), bls.B2)) is None)
    off = bytearray(bls.g2_compress(py_setup.g2[0]))
    off[:48] = (1).to_bytes(48, "big")
    off[48:] = x_off.to_bytes(48, "big")
    off[0] |= 0x80
    big_c0 = bytearray(raws[0])
    c0 = int.from_bytes(raws[0][48:], "big") + P
    big_c0[48:] = c0.to_bytes(48, "big")
    g = {"valid": raws, "sign flip": [bytes([r[0] ^ 0x20]) + r[1:] for r in raws],
         "infinity": [bytes([0xC0]) + bytes(95)], "no flag": [bytes(96), bytes([raws[0][0] & 0x7F]) + raws[0][1:]],
         "x not on curve": [bytes(off)], "x.c0 >= p": [bytes(big_c0)]}
    cases, cls = balanced(g)
    res = run_layout(hx, OP_G2_DECOMPRESS, [bytes_words(b) for b in cases], cls, 49, layout)
    for b, c, out in zip(cases, cls, res):
        try:
            want = bls.g2_decompress(b)
            status = 2 if want is None else 1
        except bls.PointError:
            want, status = None, 0
        assert out[0] == status, (c, b.hex())
        if status == 1:
            assert (_fp2_from(out[1:25]), _fp2_from(out[25:49])) == want, c
    # Fp2 inverse and square root
    qr = next(x for x in range(2, 100) if bls.fp_sqrt(x) is not None)
    nqr = next(x for x in range(2, 100) if bls.fp_sqrt(x) is None)
    sq = [bls.fp2_sqr((rnd.randrange(P), rnd.randrange(P))) for _ in range(4)]
    nsq = [a for a in ((rnd.randrange(P), rnd.randrange(1, P)) for _ in range(40)) if bls.fp2_sqrt(a) is None][:4]
    g = {"zero": [(0, 0)], "real QR": [(1, 0), (qr, 0), (4, 0)], "real non-QR": [(nqr, 0), (P - 1, 0) if bls.fp_sqrt(P - 1) is None else (nqr, 0)],
         "imaginary": [(0, 1), (0, qr), (0, nqr)], "square": sq, "non-square": nsq}
    cases, cls = balanced(g)
    recs = [_fp2_words(a) for a in cases]
    res = run_layout(hx, OP_FP2_INV, recs, cls, 24, layout)
    for a, c, out in zip(cases, cls, res):
        assert _fp2_from(out) == ((0, 0) if a == (0, 0) else bls.fp2_inv(a)), ("fp2_inv", c)
    res = run_layout(hx, OP_FP2_SQRT, recs, cls, 25, layout)
    for a, c, out in zip(cases, cls, res):
        has = bls.fp2_sqrt(a) is not None
        assert out[0] == (1 if has else 0), ("fp2_sqrt", c, a)
        if has:
            assert bls.fp2_sqr(_fp2_from(out[1:])) == a, ("fp2_sqrt", c, a)


# ------------------------------------------------------------------ SHA-256
@pytest.mark.parametrize("layout", LAYOUTS)
def test_sha256_oneshot(hx, layout):
    rnd = random.Random(71)
    lens = [0, 1, 55, 56, 63, 64, 65, 119, 120, 127, 128, 1000]
    cases = [bytes(rnd.randrange(256) for _ in range(n)) for n in lens for _ in range(3)]
    cls = [len(m) for m in cases]
    recs = [[len(m)] + bytes_words(m + bytes(-len(m) % 4)) for m in cases]
    res = run_layout(hx, OP_SHA256_ONESHOT, recs, cls, 8, layout)
    for m, out in zip(cases, res):
        assert words_bytes(out) == hashlib.sha256(m).digest(), len(m)


# block counts the library passes: verify.cu hashes (32 + 160 n) bytes of tuples for n blobs (full blocks only,
# in chunk ranges), cells_verify.cu 4 (12 + 12 commitments + 528 cells) bytes, poly.cu 2048 blocks per blob
SHA_BLOCKS = [1, 2, 31, 32, 33, 63, 64, 65] + [(32 + 160 * n) // 64 for n in (1, 2, 4, 6)] + \
             [(12 + 12 * nc + 528 * ncell) // 16 for nc, ncell in ((1, 1), (1, 2), (2, 4))] + [2048]


def test_sha256_warp_blocks(hx):
    """sha256_warp_blocks: 32 lanes expand 32 blocks, lane 0 runs the rounds; the tail branch (cnt < 32) runs
    for every count that is not a multiple of 32."""
    device_only(hx)
    rnd = random.Random(72)
    assert any(n % 32 for n in SHA_BLOCKS) and any(n % 32 == 0 for n in SHA_BLOCKS)
    msgs, recs = [], []
    for nb in SHA_BLOCKS:
        ln = 64 * nb - 9 - rnd.randrange(0, 55)
        m = bytes(rnd.randrange(256) for _ in range(ln))
        padded = m + b"\x80" + bytes((55 - ln) % 64) + (8 * ln).to_bytes(8, "big")
        assert len(padded) == 64 * nb
        msgs.append(m)
        recs.append([nb] + bytes_words(padded))
    outs = hx.run(OP_SHA256_WARP, recs, 8)
    for nb, m, out in zip(SHA_BLOCKS, msgs, outs):
        assert words_bytes(out) == hashlib.sha256(m).digest(), nb


# ------------------------------------------------------------------ pairing
def _g2_words(q):
    (x0, x1), (y0, y1) = q
    return mont_fp(x0) + mont_fp(x1) + mont_fp(y0) + mont_fp(y1)


def _fp12_flat(w):
    from tests.test_host_emul import _tower_to_flat
    vals = [canon(w[12 * i:12 * i + 12], P) * RP_INV % P for i in range(12)]
    return _tower_to_flat(b"".join(v.to_bytes(48, "big") for v in vals))


def test_pairing(hx, py_setup):
    """warp_pairing_product on one LW_PAIR_LANES-thread block (Fp12 values in shared memory) and the single-thread
    pairing of the same pairs: bit-identical Fp12 results, both equal to e(P0, Q0)^-3 e(P1, Q1)^-3 of the oracle."""
    device_only(hx)
    from oracle.py import pairing as pr

    g2_0, g2_1 = py_setup.g2[0], py_setup.g2[1]
    A = bls.g1_mul(bls.G1, 987654321)
    tA = bls.g1_mul(A, py_setup.tau)
    cases = [((tA, g2_0), (bls.g1_neg(A), g2_1), True),
             ((tA, g2_0), (A, g2_1), False),
             ((None, g2_0), (None, g2_1), True),
             ((None, g2_0), (bls.g1_neg(A), g2_1), False)]
    recs = [aff_words(p0) + aff_words(p1) + _g2_words(q0) + _g2_words(q1) for (p0, q0), (p1, q1), _ in cases]
    outs = hx.run(OP_PAIRING, recs, 290)
    for ((p0, q0), (p1, q1), one), out in zip(cases, outs):
        assert out[:144] == out[144:288], "warp and single-thread Fp12 differ"
        assert out[288] == out[289] == (1 if one else 0)
        e = pr.ONE
        for p, q in ((p0, q0), (p1, q1)):
            if p is not None:
                e = pr.mul(e, pr.pairing(p, q))
        assert pr.mul(_fp12_flat(out[:144]), pr.fpow(e, 3)) == pr.ONE
