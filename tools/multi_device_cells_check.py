#!/usr/bin/env python3
"""lwkzg_set_devices for the PeerDAS calls: ONE process, one C call, every visible GPU.  The sharded cell batch and the
sharded recovery batch must return the bytes of the single-device calls, and the sharded many-batch cell verification
their verdicts, statuses and challenges, as must the sharded verification from blobs (MODE_DENEB: the replicas get the monomial SRS from the primary context).  Prints MULTI_DEVICE_CELLS_OK on success."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import lambdaworks_kzg_b200 as lw

g = torch.cuda.device_count()
assert g >= 2, "needs at least two GPUs"
n = int(os.environ.get("NB", "512"))
lw.set_option("mode", 2)
lw.set_option("window_bits", 10)
lw.set_option("cell_window_bits", int(os.environ.get("CWB", "12")))
s = lw.load_trusted_setup_file(os.path.join(os.path.dirname(__file__), "..", "tests", "golden", "trusted_setup.txt"))
blobs = b"".join(lw.synth_blob_host(k) for k in range(n))


def run(tag):
    t0 = time.perf_counter()
    cells, proofs, st = lw.compute_cells_and_kzg_proofs_batch(blobs, n, s)
    dt = time.perf_counter() - t0
    assert not any(st)
    print("%s: %d blobs in %.1f ms (%.0f blobs/s)" % (tag, n, dt * 1e3, n / dt), flush=True)
    return cells, proofs


def recover(tag, idx, sel):
    t0 = time.perf_counter()
    cells, proofs, st = lw.recover_cells_and_kzg_proofs_batch(idx, sel, 64, n, s)
    dt = time.perf_counter() - t0
    assert not any(st)
    print("%s: recovered %d blobs from 64 cells each in %.1f ms" % (tag, n, dt * 1e3), flush=True)
    return cells, proofs


run("1 device (first call builds the FK20 tables)")
c1, p1 = run("1 device ")
keep = list(range(1, 128, 2))
idx = keep * n
sel = b"".join(c1[(b * 128 + i) * 2048: (b * 128 + i + 1) * 2048] for b in range(n) for i in keep)
rc1, rp1 = recover("1 device ", idx, sel)
assert rc1 == c1 and rp1 == p1, "recovered outputs differ from the computed ones"
# one batch per column over the first 48 blobs, plus a batch whose proof is swapped and one with an index >= 128
coms, st = lw.blob_to_kzg_commitment_batch(blobs[: 48 * 131072], 48, s)
assert not any(st)
vb = [([coms[b] for b in range(48)], [col] * 48, [c1[(b * 128 + col) * 2048: (b * 128 + col + 1) * 2048] for b in range(48)],
       [p1[(b * 128 + col) * 48: (b * 128 + col + 1) * 48] for b in range(48)]) for col in range(128)]
vb[5] = (vb[5][0], vb[5][1], vb[5][2], [vb[5][3][1], vb[5][3][0]] + vb[5][3][2:])
vb[77] = (vb[77][0], [128] + vb[77][1][1:], vb[77][2], vb[77][3])


def verify(tag):
    t0 = time.perf_counter()
    oks, sts = lw.verify_cell_kzg_proof_batches(vb, s)
    dt = time.perf_counter() - t0
    print("%s: verified %d cell batches in %.1f ms" % (tag, len(vb), dt * 1e3), flush=True)
    return oks, sts, lw.debug_cell_batch_challenges(len(vb), s)


# blob transactions of 1 to 6 blobs over the first 48 blobs, one with swapped commitments and one whose commitment
# does not decode
txs = []
for t in range(64):
    sel = [(t * 7 + j) % 48 for j in range(1 + t % 6)]
    txs.append(([blobs[b * 131072: (b + 1) * 131072] for b in sel], [coms[b] for b in sel], [p1[(b * 128 + k) * 48: (b * 128 + k + 1) * 48] for b in sel for k in range(128)]))
txs[9] = (txs[9][0], txs[9][1][::-1], txs[9][2])
txs[40] = (txs[40][0], [b"\xff" * 48] + txs[40][1][1:], txs[40][2])


def verify_blobs(tag):
    t0 = time.perf_counter()
    oks, sts = lw.verify_blob_cell_kzg_proof_batches(txs, s)
    dt = time.perf_counter() - t0
    print("%s: verified %d blob transactions in %.1f ms" % (tag, len(txs), dt * 1e3), flush=True)
    return oks, sts, lw.debug_cell_batch_challenges(len(txs), s)


v1 = verify("1 device ")
b1 = verify_blobs("1 device ")
assert b1[0] == [t not in (9, 40) for t in range(64)] and b1[1] == [lw.C_KZG_BADARGS if t == 40 else 0 for t in range(64)]
assert v1[0] == [b not in (5, 77) for b in range(128)] and v1[1] == [lw.C_KZG_BADARGS if b == 77 else 0 for b in range(128)]
lw.set_devices(list(range(g)))
run("%d devices (first call builds the replicas)" % g)
c2, p2 = run("%d devices" % g)
assert c1 == c2 and p1 == p2, "multi-device cell outputs differ from the single-device outputs"
rc2, rp2 = recover("%d devices" % g, idx, sel)
assert rc2 == rc1 and rp2 == rp1, "multi-device recovery outputs differ from the single-device outputs"
assert verify("%d devices" % g) == v1, "multi-device cell verification differs from the single-device verdicts, statuses or challenges"
assert verify_blobs("%d devices" % g) == b1, "multi-device verification from blobs differs from the single-device verdicts, statuses or challenges"
lw.set_devices([])
print("MULTI_DEVICE_CELLS_OK", flush=True)
