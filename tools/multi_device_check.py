#!/usr/bin/env python3
"""lwkzg_set_devices: ONE process, one C call per batch, every visible GPU (SURVEY §8b / §8e).  The sharded calls must
return the bytes of the single-device calls, the sharded batched verification the same boolean, and the sharded
lwkzg_verify_blob_kzg_proof_batches the single-device verdicts, statuses and challenges.  Prints MULTI_DEVICE_CHECK_OK
on success."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import lambdaworks_kzg_b200 as lw

g = torch.cuda.device_count()
assert g >= 2, "needs at least two GPUs"
n = int(os.environ.get("NB", "1536"))
B = 131072
lw.set_option("window_bits", int(os.environ.get("WB", "13")))
s = lw.load_trusted_setup_file(os.path.join(os.path.dirname(__file__), "..", "tests", "golden", "trusted_setup.txt"))
blobs = b"".join(lw.synth_blob_host(k) for k in range(n))
bl = [blobs[i * B:(i + 1) * B] for i in range(n)]


def run(tag):
    t0 = time.perf_counter(); c, p, st = lw.commit_and_prove_batch(blobs, n, s); t1 = time.perf_counter()
    assert not any(st)
    ok = lw.verify_blob_kzg_proof_batch(bl, c, p, s); t2 = time.perf_counter()
    bad = list(p); bad[n // 2] = c[0]
    okb = lw.verify_blob_kzg_proof_batch(bl, c, bad, s)
    cc, st2 = lw.blob_to_kzg_commitment_batch(blobs, n, s)
    pp, st3 = lw.compute_blob_kzg_proof_batch(blobs, b"".join(c), n, s)
    # many batches of 1-6 blobs, every seventh with a proof of another blob
    batches, o = [], 0
    while o < n:
        k = min(1 + (len(batches) % 6), n - o)
        pr = list(p[o:o + k])
        if len(batches) % 7 == 3:
            pr[0] = p[(o + k) % n]
        batches.append((bl[o:o + k], c[o:o + k], pr))
        o += k
    t3 = time.perf_counter(); oks, sts = lw.verify_blob_kzg_proof_batches(batches, s); t4 = time.perf_counter()
    rs = lw.debug_blob_batch_challenges(len(batches), s)
    print("%s: commit+prove %.1f ms, verify %.1f ms -> %s, corrupted -> %s, %d blob batches %.1f ms" %
          (tag, (t1 - t0) * 1e3, (t2 - t1) * 1e3, ok, okb, len(batches), (t4 - t3) * 1e3), flush=True)
    assert ok is True and okb is False and cc == c and pp == p
    assert oks == [i % 7 != 3 for i in range(len(batches))] and not any(sts)
    return c, p, (oks, sts, rs)


c1, p1, v1 = run("1 device ")
lw.set_devices(list(range(g)))
assert lw.get_devices() == list(range(g))
run("%d devices (first call builds the replicas)" % g)
c2, p2, v2 = run("%d devices" % g)
assert c1 == c2 and p1 == p2, "multi-device outputs differ from the single-device outputs"
assert v1 == v2, "sharded blob batches differ from the single-device call"
lw.set_devices([])
c3, p3, _ = run("1 device again")
assert c3 == c1 and p3 == p1
print("MULTI_DEVICE_CHECK_OK", flush=True)
