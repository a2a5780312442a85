"""Oracle-side helpers for the soundness tests of batched verification (CPU only, built on oracle/py).

A batched verification weights item i by r^(first + i), r the batch challenge.  A valid batch verifies under ANY
weights, and a single bad proof (or a swapped pair) fails under any weights too, so neither notices wrong weights.
What does is a pair of proofs that cancel each other out exactly when their two weights are equal.  The test setup's
secret tau (1337) is known, so such a pair is cheap: with d = tau - z (blob proofs) or d = tau^64 - h^64 (cell
proofs), proof i + aG and proof j + bG with b = -a d_i / d_j change the batch equation by a d_i (w_i - w_j) G.

Modes: 0 = MODE_REFERENCE, 1 = MODE_CKZG_LE, 2 = MODE_DENEB (the library's "mode" option).
"""
from __future__ import annotations

import hashlib
from dataclasses import dataclass
from functools import lru_cache
from typing import List, Sequence, Tuple

from oracle.py import bls, cells, kzg

R = bls.R
G = bls.G1
TORSION3 = (0, 2)   # on the curve (0^3 + 4 = 2^2), order 3: not in G1
DEFAULT_A = 0x5EED_F0E6_E5  # the multiple of G added to the first proof of a forged pair


def oracle_for(mode: int, setup: kzg.Setup):
    return (kzg.RefMode, kzg.LeMode, kzg.DenebMode)[mode](setup)


def fe_bytes(mode: int, v: int) -> bytes:
    """A field element as the mode puts it in a blob: little-endian in MODE_CKZG_LE, big-endian otherwise."""
    return (v % R).to_bytes(32, "little" if mode == 1 else "big")


def random_blob(mode: int, rnd) -> bytes:
    return b"".join(fe_bytes(mode, rnd.randrange(R)) for _ in range(kzg.FIELD_ELEMENTS_PER_BLOB))


def non_g1_points() -> List[bytes]:
    """Two compressed points on the curve but outside G1: the 3-torsion point (0, 2), and G plus it."""
    return [bls.g1_compress(TORSION3), bls.g1_compress(bls.g1_add(G, TORSION3))]


def decode_error_code(mode: int) -> int:
    """What the mode's decoder returns for a point outside G1 (C_KZG_ERROR in MODE_REFERENCE, else C_KZG_BADARGS)."""
    return kzg.C_KZG_ERROR if mode == 0 else kzg.C_KZG_BADARGS


# ------------------------------------------------------------------ blob items
@lru_cache(maxsize=4)
def _lagrange_at(x: int) -> Tuple[int, ...]:
    """L_k(x) over the bit-reversed 4096th roots of unity (x outside the domain): p(x) = sum e_k L_k(x)."""
    dom = kzg.brp_domain()
    n = len(dom)
    inv = kzg.batch_inv([(x - w) % R for w in dom])
    f = (pow(x, n, R) - 1) * bls.fr_inv(n) % R
    return tuple(w * iv % R * f % R for w, iv in zip(dom, inv))


def poly_at(o, blob: bytes, x: int) -> int:
    """The blob's polynomial at x, in the oracle's mode (coefficient form in MODE_REFERENCE)."""
    if isinstance(o, kzg.LeMode):   # DenebMode too
        evals = o.blob_to_evals(blob)
        if x == o.s.tau:   # the one point every item is evaluated at: weights computed once
            return sum(e * l for e, l in zip(evals, _lagrange_at(x))) % R
        return o.eval_at(evals, x)
    return kzg.horner(o.blob_to_coeffs(blob), x)


def challenge(o, blob: bytes, commitment: bytes) -> int:
    """Fiat-Shamir z of (blob, commitment); independent of the proof."""
    if isinstance(o, kzg.LeMode):
        return o.compute_challenge(blob, commitment)
    return o.compute_challenge(blob, bls.g1_decompress(commitment))


@dataclass
class Item:
    """A valid (blob, commitment, proof) with z, y = p(z) and the discrete logs (base G) of commitment and proof."""
    blob: bytes
    commitment: bytes
    proof: bytes
    z: int
    y: int
    c_log: int
    pi_log: int


def make_item(o, blob: bytes) -> Item:
    tau = o.s.tau
    c_log = poly_at(o, blob, tau)
    commitment = bls.g1_compress(bls.g1_mul(G, c_log))
    z = challenge(o, blob, commitment)
    y = poly_at(o, blob, z)
    pi_log = (c_log - y) * bls.fr_inv((tau - z) % R) % R
    return Item(blob, commitment, bls.g1_compress(bls.g1_mul(G, pi_log)), z, y, c_log, pi_log)


def forge_pair(proof_i: bytes, proof_j: bytes, d_i: int, d_j: int, a: int = DEFAULT_A) -> Tuple[bytes, bytes]:
    """(proof_i + aG, proof_j + bG) with b = -a d_i / d_j: the batch equation moves by a d_i (w_i - w_j) G, so the
    pair passes exactly when the two weights are equal.  d = tau - z for blob proofs (blob_factor), tau^64 - h_k^64
    for cell proofs (cell_factor)."""
    b = (-a * d_i * bls.fr_inv(d_j % R)) % R
    pi = bls.g1_add(bls.g1_decompress(proof_i), bls.g1_mul(G, a % R))
    pj = bls.g1_add(bls.g1_decompress(proof_j), bls.g1_mul(G, b))
    return bls.g1_compress(pi), bls.g1_compress(pj)


def blob_factor(o, blob: bytes, commitment: bytes) -> int:
    return (o.s.tau - challenge(o, blob, commitment)) % R


def cell_factor(tau: int, cell_index: int) -> int:
    n = cells.FIELD_ELEMENTS_PER_CELL
    return (pow(tau, n, R) - pow(cells.coset_shift_for_cell(cell_index), n, R)) % R


def forge_blob_batch(o, blobs, commitments, proofs, i: int, j: int, a: int = DEFAULT_A) -> List[bytes]:
    """The proofs of a batch with the pair (i, j) forged."""
    out = list(proofs)
    out[i], out[j] = forge_pair(proofs[i], proofs[j], blob_factor(o, blobs[i], commitments[i]), blob_factor(o, blobs[j], commitments[j]), a)
    return out


def weighted_batch_check(o, blobs, commitments, proofs, weights) -> bool:
    """The batch equation with caller-chosen weights, toxic-waste form of the 2-pairing check:
    sum w_i (C_i - y_i G + z_i pi_i) == tau sum w_i pi_i."""
    lhs, rhs = None, None
    for blob, c, p, w in zip(blobs, commitments, proofs, weights):
        cp, pp = bls.g1_decompress(c), bls.g1_decompress(p)
        z = challenge(o, blob, c)
        y = poly_at(o, blob, z)
        term = bls.g1_add(bls.g1_add(cp, bls.g1_neg(bls.g1_mul(G, y))), bls.g1_mul(pp, z))
        lhs = bls.g1_add(lhs, bls.g1_mul(term, w % R))
        rhs = bls.g1_add(rhs, bls.g1_mul(pp, w % R))
    return lhs == bls.g1_mul(rhs, o.s.tau)


# ------------------------------------------------------------------ phase 1 / 2 / 3 of the library's layout
def batch_challenge(mode: int, commitments: Sequence[bytes], zs: Sequence[int], ys: Sequence[int], proofs: Sequence[bytes]) -> int:
    """r = H(domain || 4096 || n || (C_i || z_i || y_i || pi_i)...).  MODE_REFERENCE: 8-byte little-endian counts,
    big-endian field elements, digest read big-endian; MODE_CKZG_LE: everything little-endian; MODE_DENEB:
    everything big-endian."""
    hdr = "big" if mode == 2 else "little"
    msg = kzg.RANDOM_CHALLENGE_KZG_BATCH_DOMAIN + kzg.FIELD_ELEMENTS_PER_BLOB.to_bytes(8, hdr) + len(commitments).to_bytes(8, hdr)
    msg += tuples(mode, commitments, zs, ys, proofs)
    return int.from_bytes(hashlib.sha256(msg).digest(), "little" if mode == 1 else "big") % R


def tuples(mode: int, commitments, zs, ys, proofs) -> bytes:
    """Phase-1 output: 160 bytes per item, C || z || y || pi with z, y in the mode's byte order."""
    return b"".join(c + fe_bytes(mode, z) + fe_bytes(mode, y) + p for c, z, y, p in zip(commitments, zs, ys, proofs))


def items_challenge(mode: int, items: Sequence[Item]) -> int:
    return batch_challenge(mode, [t.commitment for t in items], [t.z for t in items], [t.y for t in items], [t.proof for t in items])


def items_tuples(mode: int, items: Sequence[Item]) -> bytes:
    return tuples(mode, [t.commitment for t in items], [t.z for t in items], [t.y for t in items], [t.proof for t in items])


def _be96(pt) -> bytes:
    return bytes(96) if pt is None else pt[0].to_bytes(48, "big") + pt[1].to_bytes(48, "big")


def _from_be96(b: bytes):
    return None if not any(b) else (int.from_bytes(b[:48], "big"), int.from_bytes(b[48:], "big"))


def expected_partial(items: Sequence[Item], r: int, first: int) -> bytes:
    """Phase-2 output of the items [first, first + len(items)) of a batch with challenge r: three 96-byte big-endian
    uncompressed points (all zeros = infinity)
        sum w_i pi_i  |  96 zero bytes  |  sum w_i z_i pi_i + sum w_i C_i - (sum w_i y_i) G,    w_i = r^(first + i)
    each computed from the discrete logs with one scalar multiplication."""
    s1 = s3 = 0
    for k, t in enumerate(items):
        w = pow(r, first + k, R)
        s1 += w * t.pi_log
        s3 += w * (t.z * t.pi_log + t.c_log - t.y)
    return _be96(bls.g1_mul(G, s1 % R)) + bytes(96) + _be96(bls.g1_mul(G, s3 % R))


def phase3(partials: bytes, tau: int) -> bool:
    """The library's phase 3 in toxic-waste form: with A = sum of the second and third points of every partial and
    B = sum of the first ones, e(A, G2) == e(B, [tau] G2)."""
    a = b = None
    for off in range(0, len(partials), 288):
        p = partials[off: off + 288]
        b = bls.g1_add(b, _from_be96(p[:96]))
        a = bls.g1_add(bls.g1_add(a, _from_be96(p[96:192])), _from_be96(p[192:]))
    return a == bls.g1_mul(b, tau)


# ------------------------------------------------------------------ cells
def cell_interp_at(co: cells.CellOracle, cell: bytes, cell_index: int, x: int) -> int:
    """I_k(x): the polynomial of degree < 64 through the cell's evaluations on its coset."""
    n = cells.FIELD_ELEMENTS_PER_CELL
    a = cells.ifft(cells.brp(co.cell_to_evals(cell)), cells.root_of_unity(n))
    t = x * bls.fr_inv(cells.coset_shift_for_cell(cell_index)) % R
    return kzg.horner(a, t)


def weighted_cell_check(co: cells.CellOracle, commitments, cell_indices, cell_bytes, proofs, weights) -> bool:
    """verify_cell_kzg_proof_batch with caller-chosen weights (toxic-waste form):
    sum w_k (C_k - I_k(tau) G + h_k^64 pi_k) == tau^64 sum w_k pi_k."""
    n = cells.FIELD_ELEMENTS_PER_CELL
    tau = co.s.tau
    lhs, rhs = None, None
    decoded = {c: bls.g1_decompress(c) for c in set(commitments)}
    for c, k, cell, p, w in zip(commitments, cell_indices, cell_bytes, proofs, weights):
        pp = bls.g1_decompress(p)
        h64 = pow(cells.coset_shift_for_cell(k), n, R)
        s = (w * -cell_interp_at(co, cell, k, tau)) % R
        term = bls.g1_add(bls.g1_add(bls.g1_mul(decoded[c], w % R), bls.g1_mul(G, s)), bls.g1_mul(pp, w * h64 % R))
        lhs = bls.g1_add(lhs, term)
        rhs = bls.g1_add(rhs, bls.g1_mul(pp, w % R))
    return lhs == bls.g1_mul(rhs, pow(tau, n, R))


def forge_cell_batch(tau: int, cell_indices, proofs, i: int, j: int, a: int = DEFAULT_A) -> List[bytes]:
    out = list(proofs)
    out[i], out[j] = forge_pair(proofs[i], proofs[j], cell_factor(tau, cell_indices[i]), cell_factor(tau, cell_indices[j]), a)
    return out
