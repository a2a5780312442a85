"""GPU tier: the three MSMs behind almost every output -- the FK20 gather of the cell proofs, the commitment / blob-proof
gather and the variable-base bucket MSM -- at every window the library can pick at run time, not only the ones the
other modules pin.

The window of each one is a run-time choice (a default, what free HBM allows, or n), and the kernels change shape
with it: empty accumulator slots and a partial last round in the batched-affine kernel, a top window of a different
size in the digit tables, several reduction blocks per window and a 2^16-bucket top window in the bucket MSM.

The setup is the monomial tau = 1337 one, so every SRS point has a known discrete log: the expected value of an MSM
over SRS points is one [sum s_i dlog_i] G.  Outputs do not depend on the window, so every window's bytes are also
compared with the bytes at window 8, computed once per module.
"""
import contextlib
import os
import random
from collections import Counter

import pytest

from oracle.py import bls, kzg
from tests import _forge
from tests.golden.make_cell_fixtures import make_blob

pytestmark = pytest.mark.gpu

SETUP = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "trusted_setup.txt")
R = bls.R
B = kzg.BYTES_PER_BLOB
TAU = 1337
X2 = bls.BLS_X ** 2                    # GLV split modulus: k = m + q x^2
INF = bytes([0xC0]) + bytes(47)
GIB = 1 << 30
OPTIONS = ("mode", "window_bits", "cell_window_bits", "cell_chunk_blobs", "msm_algo", "msm_ba_min_blobs", "msm_ba_variant",
           "lincomb_points_in_g1", "share_table")
VM_HOOKS = ("LWKZG_VM_C", "LWKZG_VM_GLV", "LWKZG_VM_S")
CELL_WINDOWS = list(range(4, 15))
COMMIT_WINDOWS = [4, 5, 6, 7, 9, 10, 11, 12, 14, 15]      # 8, 13 and 16 are pinned by other modules
PARTIAL_ROUND_WINDOWS = [7, 12, 14, 15]                   # batched-affine rounds that end part-filled
KERNELS = [("xyzz", dict(msm_algo=0)),
           ("batched-affine v0", dict(msm_algo=1, msm_ba_min_blobs=1, msm_ba_variant=0)),
           ("batched-affine v1", dict(msm_algo=1, msm_ba_min_blobs=1, msm_ba_variant=1))]


@pytest.fixture(scope="module")
def lw():
    import lambdaworks_kzg_b200 as m

    m.load_library()
    return m


@pytest.fixture(scope="module")
def start_options(lw):
    """Every option this module changes, as the module found it."""
    return {k: lw.get_option(k) for k in OPTIONS}


@pytest.fixture(autouse=True)
def _options_and_hooks_restored(lw, start_options):
    assert not any(h in os.environ for h in VM_HOOKS)
    yield
    assert {k: lw.get_option(k) for k in OPTIONS} == start_options
    assert not any(h in os.environ for h in VM_HOOKS), "a LWKZG_VM_* hook outlived its call"


@contextlib.contextmanager
def _options(lw, start, **kv):
    try:
        for k, v in kv.items():
            lw.set_option(k, v)
        yield
    finally:
        for k in kv:
            lw.set_option(k, start[k])


@contextlib.contextmanager
def _settings(lw, start, **kv):
    """One settings object at a time, private table (no IPC handle, nothing under /dev/shm), freed on every exit."""
    with _options(lw, start, share_table=0, **kv):
        s = lw.load_trusted_setup_file(SETUP)
        try:
            yield s
        finally:
            s.free()


def _table_bytes(lw, c):
    """Bytes of one digit table of 4096 points at window c (the commitment table; the FK20 table is two of them)."""
    _, counts = lw.table_geometry(c)
    return 4096 * sum(counts) * 96


def _skip_unless_free(need, what):
    import torch

    free, _ = torch.cuda.mem_get_info()
    if free < need + 8 * GIB:
        pytest.skip("%s needs %d bytes + 8 GiB, %d bytes free" % (what, need, free))


def _first_diff(a, b, each=48):
    for i in range(0, min(len(a), len(b)), each):
        if a[i: i + each] != b[i: i + each]:
            return i // each
    return None if len(a) == len(b) else "length"


# ------------------------------------------------------------------ A. FK20 cell proofs at every cell window
def _cell_edge_blobs(lw):
    return [make_blob(61, 2), make_blob(62, 2),
            bytes(B),                                               # zero polynomial
            (5).to_bytes(32, "big") * 4096,                         # constant
            (3).to_bytes(32, "big") + bytes(32 * 4095),             # one non-zero word, first
            bytes(32 * 4095) + (3).to_bytes(32, "big"),             # one non-zero word, last
            (R - 1).to_bytes(32, "big") * 4096,
            lw.synth_blob_host(7)]


def _cell_batch(lw, edge, n):
    """n blobs for one pass of the segmented batched-affine kernel: the edge blobs at the start, in the middle and at
    the end, synthetic blobs elsewhere."""
    blobs = [lw.synth_blob_host(2000 + k) for k in range(n)]
    m = n // 2 - len(edge) // 2
    blobs[: len(edge)] = edge
    blobs[m: m + len(edge)] = edge[3:] + edge[:3]
    blobs[n - len(edge):] = edge[::-1]
    return b"".join(blobs)


def _cell_proofs(lw, s, blobs, n, chunk, want_cells=False):
    lw.set_option("cell_chunk_blobs", chunk)
    cells, proofs, st = lw.compute_cells_and_kzg_proofs_batch(blobs, n, s, want_cells=want_cells)
    assert st == [0] * n
    return cells, proofs


@pytest.fixture(scope="module")
def cell_edge(lw):
    return _cell_edge_blobs(lw)


@pytest.fixture(scope="module")
def cell_ref8(lw, start_options, cell_edge):
    """Proof bytes at cell window 8 (what the other cell modules pin): the edge blobs on the warp kernel, 224 and 230
    blobs on the segmented batched-affine kernel."""
    with _settings(lw, start_options, mode=2, window_bits=8, cell_window_bits=8, cell_chunk_blobs=888) as s:
        out = {"edge": _cell_proofs(lw, s, b"".join(cell_edge), len(cell_edge), 888)[1]}
        assert lw.cell_window_bits(s) == 8
        for n in (224, 230):
            out[n] = _cell_proofs(lw, s, _cell_batch(lw, cell_edge, n), n, 888)[1]
    # the degenerate blobs anchor the reference: zero and constant polynomials have infinity proofs
    assert out["edge"][2 * 6144: 4 * 6144] == INF * 256
    return out


@pytest.fixture(scope="module")
def o2(py_setup):
    from oracle.py import cells

    return cells.CellOracle(py_setup, 2)


def _check_fk20_stages(lw, s, o2):
    """The FK20 intermediates against the exponent model (tau known), so that a failure names its stage."""
    from oracle.py import cells
    from oracle.py.kzg import _bitrev

    blob = make_blob(41, 2)
    f = o2.blob_to_coeffs(blob)
    scalars, hhat, h, fk = lw.debug_cell_stages(blob, s)
    nu = pow(cells.root_of_unity(8192), 64, R)
    sp = [pow(TAU, k, R) for k in range(4096)]
    inv128 = bls.fr_inv(128)
    X, C = [], []
    for b in range(64):
        X.append(cells.fft([sp[64 * (62 - v) + b] if v <= 62 else 0 for v in range(128)], nu))
        c = [0] * 128
        c[0] = f[64 * 63 + b]
        for u in range(66, 128):
            c[u] = f[64 * (u - 65) + b]
        C.append(cells.fft(c, nu))
    assert all(scalars[j * 64 + b] == C[b][j] * inv128 % R for j in range(128) for b in range(64)), "MSM scalars"
    rng = random.Random(2)
    for j, b in [(0, 0), (64, 5), (127, 63)] + [(rng.randrange(128), rng.randrange(64)) for _ in range(40)]:
        assert fk[j * 64 + b] == bls.g1_mul(bls.G1, X[b][j]), ("FK20 points", j, b)
    hh = [sum(C[b][j] * X[b][j] for b in range(64)) * inv128 % R for j in range(128)]
    for j in range(128):
        assert hhat[j] == bls.g1_compress(bls.g1_mul(bls.G1, hh[j])), ("MSM result", j)
    H = cells.fft(hh, bls.fr_inv(nu))
    for p in range(128):
        want = bls.g1_mul(bls.G1, H[_bitrev(p, 7)]) if p % 2 == 0 else None
        assert h[p] == bls.g1_compress(want), ("inverse G1 FFT", p)


@pytest.mark.parametrize("c", CELL_WINDOWS)
def test_fk20_cell_proofs_at_cell_window(lw, start_options, cell_edge, cell_ref8, o2, c):
    """FK20 cell proofs with the digit table at window c: the warp-per-frequency kernel (passes below 224 blobs) and
    the segmented batched-affine kernel (224 and 230 blobs in one pass) give the window-8 bytes."""
    with _settings(lw, start_options, mode=2, window_bits=8, cell_window_bits=c, cell_chunk_blobs=888) as s:
        _skip_unless_free(2 * _table_bytes(lw, c), "the FK20 table at window %d" % c)
        edge = _cell_proofs(lw, s, b"".join(cell_edge), len(cell_edge), 888)[1]
        assert lw.cell_window_bits(s) == c
        assert edge == cell_ref8["edge"], ("warp kernel", _first_diff(edge, cell_ref8["edge"]))
        if c in (7, 13):
            coeffs = o2.blob_to_coeffs(cell_edge[0])
            for k in range(128):
                assert edge[48 * k: 48 * k + 48] == bls.g1_compress(o2.proof_for_cell(coeffs, k)), k
        for n in (224, 230):
            blobs = _cell_batch(lw, cell_edge, n)
            cells, big = _cell_proofs(lw, s, blobs, n, 888, want_cells=(c == 13 and n == 230))
            _, warp = _cell_proofs(lw, s, blobs, n, 100)
            lw.set_option("cell_chunk_blobs", 888)
            assert big == warp, ("batched-affine vs warp", n, _first_diff(big, warp))
            assert big == cell_ref8[n], ("batched-affine vs window 8", n, _first_diff(big, cell_ref8[n]))
        if c == 13:
            _check_fk20_stages(lw, s, o2)
            coms, st = lw.blob_to_kzg_commitment_batch(blobs, 230, s)
            assert st == [0] * 230
            rng = random.Random(13)
            pick = [(b, rng.randrange(128)) for b in range(0, 230, 3)] + [(2, 5), (229, 127), (115, 0)]
            cell = lambda b, i: cells[(b * 128 + i) * 2048: (b * 128 + i + 1) * 2048]  # noqa: E731
            proof = lambda b, i: big[(b * 128 + i) * 48: (b * 128 + i + 1) * 48]  # noqa: E731
            args = ([coms[b] for b, _ in pick], [i for _, i in pick], [cell(b, i) for b, i in pick], [proof(b, i) for b, i in pick])
            assert lw.verify_cell_kzg_proof_batch(*args, s) is True
            pr = list(args[3])
            pr[10], pr[11] = pr[11], pr[10]
            assert lw.verify_cell_kzg_proof_batch(args[0], args[1], args[2], pr, s) is False


# ------------------------------------------------------------------ B. commitment and blob proof at the fallback windows
def blob_from_coeffs(coeffs):
    b = b"".join((c % (1 << 256)).to_bytes(32, "big") for c in coeffs)
    return b + bytes(B - len(b))


def edge_blobs():
    rnd = random.Random(4844)
    return {
        "zero": bytes(B),
        "one": blob_from_coeffs([1]),
        "x": blob_from_coeffs([0, 1]),
        "top_only": blob_from_coeffs([0] * 4095 + [7]),
        "all_ff": b"\xff" * B,                                  # every word >= r (reduced mod r)
        "r_minus_1": blob_from_coeffs([R - 1] * 4096),
        "exactly_r": blob_from_coeffs([R] * 4096),               # == all-zero polynomial
        "r_plus_1": blob_from_coeffs([R + 1, 2 * R + 3, 2 * R - 1] + [0] * 10 + [R]),
        "random_full": bytes(rnd.randrange(256) for _ in range(B)),
        "sparse": blob_from_coeffs([rnd.randrange(R) if i % 97 == 0 else 0 for i in range(4096)]),
        "repeat_digit": blob_from_coeffs([0x0101010101010101010101010101010101010101010101010101010101010101 % R] * 4096),
    }


@pytest.fixture(scope="module")
def ref(py_setup):
    return kzg.RefMode(py_setup)


@pytest.fixture(scope="module")
def edge_ref(ref):
    out = {}
    for name, blob in edge_blobs().items():
        c = ref.blob_to_kzg_commitment(blob)
        out[name] = (c, ref.compute_blob_kzg_proof(blob, c))
    return out


@pytest.fixture(scope="module")
def synth_ref(lw, ref):
    memo = {}

    def get(k):
        if k not in memo:
            blob = lw.synth_blob_host(k)
            c = ref.blob_to_kzg_commitment(blob)
            memo[k] = (c, ref.compute_blob_kzg_proof(blob, c))
        return memo[k]
    return get


@pytest.mark.parametrize("c", COMMIT_WINDOWS)
def test_commitment_and_blob_proof_at_window(lw, start_options, edge_ref, synth_ref, c):
    """commit_and_prove_batch with the commitment table at window c, on the XYZZ kernel and both batched-affine
    variants: the edge blobs against the oracle, and at the windows whose batched-affine rounds end part-filled,
    batches of 1, 60, 120 and 230 blobs (8, 4, 2 and 1 blocks per blob)."""
    _skip_unless_free(_table_bytes(lw, c), "the commitment table at window %d" % c)
    blobs = edge_blobs()
    names = list(blobs)
    cat = b"".join(blobs[n] for n in names)
    with _settings(lw, start_options, mode=0, window_bits=c) as s:
        assert lw.window_bits(s) == c

        def run(kernel, data, n):
            with _options(lw, start_options, **kernel):
                coms, proofs, st = lw.commit_and_prove_batch(data, n, s)
            assert st == [0] * n
            return coms, proofs

        for kname, kernel in KERNELS:
            coms, proofs = run(kernel, cat, len(names))
            for i, name in enumerate(names):
                assert (coms[i], proofs[i]) == edge_ref[name], (kname, name)
        if c in PARTIAL_ROUND_WINDOWS:
            for n in (1, 60, 120, 230):
                data = b"".join(lw.synth_blob_host(k) for k in range(n))
                outs = [run(kernel, data, n) for _, kernel in KERNELS]
                for (kname, _), out in zip(KERNELS[1:], outs[1:]):
                    assert out == outs[0], (kname, n, [k for k in range(n) if (out[0][k], out[1][k]) != (outs[0][0][k], outs[0][1][k])][:5])
                for k in sorted({0, n // 2, n - 1}):
                    assert (outs[0][0][k], outs[0][1][k]) == synth_ref(k), (n, k)


# ------------------------------------------------------------------ C. variable-base MSM: every plan
def _enc(p):
    return bytes(96) if p is None else p[0].to_bytes(48, "big") + p[1].to_bytes(48, "big")


def _vm_plan(n, c, glv, s_force):
    """Host mirror of vm_layout / vm_run (csrc/varmsm.cu): windows, buckets per signed window, lanes per bucket and the
    run length above which a bucket goes to vm_heavy_kernel."""
    items = 2 * n if glv else n
    w = -(-(128 if glv else 255) // c)
    nb_half = 1 << (c - 1)
    avg = items // nb_half + 1
    s = 1
    while s < 32 and (w + 1) * nb_half * 2 * s <= 592 * 32 * 6 and 2 * s * 4 <= avg:
        s <<= 1
    s = s_force or s
    return w, s, min(max(4 * avg, 16 * s), 384 * s)


def _vm_bucket_counts(scalars, c, glv):
    """Entries per (window, bucket) as the device's signed-digit recoding produces them (unsigned top window)."""
    w = -(-(128 if glv else 255) // c)
    cnt = Counter()
    for k in scalars:
        k %= R
        for h in ((k % X2, k // X2) if glv else (k,)):
            carry = 0
            for j in range(w):
                d = ((h >> (c * j)) & ((1 << c) - 1)) + carry
                carry = 0
                if j < w - 1 and d > 1 << (c - 1):
                    d -= 1 << c
                    carry = 1
                if d:
                    cnt[(j, abs(d) - 1)] += 1
    return cnt


def _boundary_values(c, bits):
    """Values whose c-bit digits sit on the recoding's edges at every window position: the largest positive digit,
    one more (a carry), and runs of ones that carry through every window into the top one."""
    w = -(-bits // c)
    vals = []
    for j in range(w):
        vals.append((1 << (c - 1)) << (c * j))
        vals.append(((1 << (c - 1)) + 1) << (c * j))
        vals.append((1 << (c * (j + 1))) - 1)
    return vals


def _boundary_scalars(c, glv):
    if not glv:
        sc = [v for v in _boundary_values(c, 255) if v < 1 << 256]
    else:
        hv = [v for v in _boundary_values(c, 128) if v < X2] + [(1 << 127) - 1, X2 - 1]
        sc = hv + [v * X2 for v in hv] + [hv[i] + hv[(i + 1) % len(hv)] * X2 for i in range(len(hv))]
        q_max = (R - X2) // X2            # largest q with m = x^2 - 1 and k < r
        sc += [X2 - 1 + q_max * X2, (X2 - 1 + (X2 - 2) * X2) % R]
        sc = [k if k < 1 << 256 else k % R for k in sc]
    return sc + [R - 1, R, R + 1, 0]


@pytest.fixture(scope="module")
def srs(py_setup):
    """(encoded points, discrete logs) of the 4096 SRS points: point i is tau^i G."""
    assert py_setup.tau == TAU
    return [_enc(p) for p in py_setup.g1], [pow(TAU, i, R) for i in range(4096)]


def _case(srs, idx, scalars, name):
    pts, dl = srs
    acc = sum((s % R) * dl[i] for i, s in zip(idx, scalars)) % R
    return (name, b"".join(pts[i] for i in idx), b"".join(s.to_bytes(32, "big") for s in scalars), len(idx),
            bls.g1_compress(bls.g1_mul(bls.G1, acc)))


HEAVY_N = 2100
HEAVY_SCALAR = random.Random(21).getrandbits(126) * (1 + X2)   # GLV halves m == q: both land in the same buckets


@pytest.fixture(scope="module")
def vm_cases(srs, py_setup):
    """Inputs whose expected value does not depend on the plan: (name, points, scalars, n, expected compressed)."""
    rng = random.Random(1337)
    cases = []
    for n in (1, 37, 300):
        cases.append(_case(srs, rng.sample(range(4096), n), [rng.getrandbits(256) for _ in range(n)], "random n=%d" % n))
    cases.append(_case(srs, list(range(HEAVY_N)), [HEAVY_SCALAR] * HEAVY_N, "equal scalars"))
    # P with -P at equal scalars (cancellation in a bucket), one point three times (doubling), infinity points
    pa, pb, pc = py_setup.g1[11], py_setup.g1[12], py_setup.g1[13]
    s1, s2, s3 = (rng.getrandbits(255) for _ in range(3))
    pts = [pa, bls.g1_neg(pa), pb, None, pb, pb, pc, None, pa]
    sc = [s1, s1, s2, s3, s2, s2, s3, 0, R - 1]
    want = bls.g1_compress(bls.g1_sum(bls.g1_mul(p, k % R) for p, k in zip(pts, sc)))
    cases.append(("cancel / double / infinity", b"".join(_enc(p) for p in pts), b"".join(k.to_bytes(32, "big") for k in sc), len(pts), want))
    cases.append(("n = 0", b"", b"", 0, INF))
    return cases


def _point_any(b):
    """Decompress a point on the curve without the subgroup check."""
    x = int.from_bytes(bytes([b[0] & 0x1F]) + b[1:], "big")
    y = bls.fp_sqrt(x * x * x + 4)
    lo, hi = sorted((y, bls.P - y))
    return (x, hi if b[0] & 0x20 else lo)


@pytest.fixture(scope="module")
def non_g1_case(py_setup):
    """The two on-curve points outside G1 among G1 points (GLV off only): [k]P with no reduction by P's order, the
    scalars still reduced mod r first as the reference does."""
    rng = random.Random(3)
    outside = [_point_any(b) for b in _forge.non_g1_points()]
    pts = [outside[0], py_setup.g1[100], outside[1], py_setup.g1[7], outside[0]]
    sc = [rng.getrandbits(256), rng.getrandbits(256), R + 2, R - 1, 5]
    want = bls.g1_compress(bls.g1_sum(bls.g1_mul(p, k % R) for p, k in zip(pts, sc)))
    return ("points outside G1", b"".join(_enc(p) for p in pts), b"".join(k.to_bytes(32, "big") for k in sc), len(pts), want)


def _lincomb(lw, monkeypatch, case, c, s_force):
    """g1_lincomb with the plan forced through the LWKZG_VM_* hooks, which are set for this one call only."""
    _, pb, sb, n, _ = case
    with monkeypatch.context() as m:
        m.setenv("LWKZG_VM_C", str(c))
        if s_force:
            m.setenv("LWKZG_VM_S", str(s_force))
        return lw.g1_lincomb(pb, sb, n)


@pytest.mark.parametrize("glv", [0, 1])
@pytest.mark.parametrize("c", list(range(4, 17)))
def test_var_msm_plan(lw, start_options, monkeypatch, srs, vm_cases, non_g1_case, c, glv):
    """Every bucket-MSM plan forced at small n: window c (with it 1 .. 64 reduction blocks per window and the
    unsigned top window), GLV split off / on, lanes per bucket S = default, 1, 4, 32."""
    sc = _boundary_scalars(c, glv)
    cases = list(vm_cases) + [_case(srs, list(range(3000, 3000 + len(sc))), sc, "digit boundaries")]
    if not glv:
        cases.append(non_g1_case)
    for s_force in (0, 1, 4, 32):
        # the equal-scalar case must send buckets to vm_heavy_kernel under this plan: its HEAVY_N scalars all fill
        # the buckets one of them fills
        _, _, cap = _vm_plan(HEAVY_N, c, glv, s_force)
        assert max(_vm_bucket_counts([HEAVY_SCALAR], c, glv).values()) * HEAVY_N > cap, (c, glv, s_force, cap)
        with _options(lw, start_options, lincomb_points_in_g1=glv):
            got = [_lincomb(lw, monkeypatch, case, c, s_force) for case in cases]
        for case, g in zip(cases, got):
            assert g == case[4], (case[0], "c", c, "glv", glv, "S", s_force or "default")


def _synth_scalar(seed, t):
    """Scalar t of bench_var_msm's synthetic input (csrc/varmsm.cu vm_synth_kernel)."""
    M = (1 << 64) - 1
    st = 0xB2004844 ^ ((seed * 4096 + t) & M)
    w = b""
    for _ in range(4):
        st = (st + 0x9E3779B97F4A7C15) & M
        z = st
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M
        w += (z ^ (z >> 31)).to_bytes(8, "big")
    return int.from_bytes(bytes([w[0] & 0x3F]) + w[1:], "big")


def test_var_msm_default_plans_at_large_n(lw, start_options, srs):
    """The plans the sizes pick by themselves: GLV at 2^17 points (window 15, the window of the 2n + 1-point MSMs of
    batched verification from 65536 blobs), and no GLV at 2^17 and 2^19 points (windows 14 and 16)."""
    n = 1 << 17
    with _settings(lw, start_options, mode=0, window_bits=8) as s:
        _, got = lw.bench_var_msm(n, s, iters=1, seed=3)
        dl = lw.synth_point_dlogs(s, n, TAU)
    acc = sum(_synth_scalar(3, t) * dl[t] for t in range(n)) % R
    assert got == bls.g1_compress(bls.g1_mul(bls.G1, acc))
    pts, dlog = srs
    rng = random.Random(19)
    for lg in (17, 19):
        n = 1 << lg
        sc = [rng.getrandbits(256) for _ in range(n)]
        per = [0] * 4096
        for i, k in enumerate(sc):
            per[i & 4095] += k
        acc = sum(p % R * d for p, d in zip(per, dlog)) % R
        with _options(lw, start_options, lincomb_points_in_g1=0):
            got = lw.g1_lincomb(b"".join(pts) * (n // 4096), b"".join(k.to_bytes(32, "big") for k in sc), n)
        assert got == bls.g1_compress(bls.g1_mul(bls.G1, acc)), lg
