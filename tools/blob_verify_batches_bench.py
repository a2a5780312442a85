#!/usr/bin/env python3
"""K blob-proof batches per call, lwkzg_verify_blob_kzg_proof_batches[_device], against K calls of the aggregate
verify_blob_kzg_proof_batch over the same batches.

MODE_DENEB, the test setup's tables at window 8.  Inputs: synthetic blobs (lwkzg_synth_blobs_device) with commitments
and proofs from lwkzg_commit_and_prove_batch_device.  Shapes K x n_b: a transaction pool's 128 transactions of 6
blobs, 32 of 6, one of 6, 4096 one-blob batches and one batch of 4096 blobs.  Arms, every one over the same batches:
  new_device    lwkzg_verify_blob_kzg_proof_batches_device, device-resident (CUDA events around the call)
  new_pinned    lwkzg_verify_blob_kzg_proof_batches from pinned host memory (host clock around the synchronous call)
  loop_device   K calls of lwkzg_verify_blob_kzg_proof_batch_device (host clock)
  loop_pinned   K calls of verify_blob_kzg_proof_batch from pinned host memory (host clock)
Median and spread of --reps repetitions after a warm-up (loops over more than 256 calls: --loop-reps).  The verdicts
are checked against the known answer (every batch true) on every arm.  A profiler run of the new call at 128 x 6
gives its per-stage kernel times.  Card name and power limit are read in the same run.

python tools/blob_verify_batches_bench.py [--reps 7] [--loop-reps 2] [--out FILE]"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import lambdaworks_kzg_b200 as lw  # noqa: E402

SHAPES = [(128, 6), (32, 6), (1, 6), (4096, 1), (1, 4096)]
BLOB = 4096 * 32
# kernel name fragments of the stages of one pass
STAGES = {
    "decode": ("g1_decompress",),
    "blob_hash_and_eval": ("challenge_midstate", "challenge_finish", "poly_eval", "le_eval", "le_blob_check", "make_tuples"),
    "batch_hashes": ("blob_batches_challenge",),
    "msm": ("blob_batches_scalars", "blob_batches_terms", "blob_batches_reduce"),
    "pairing": ("batch_final",),
}


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[-1] if q.stdout.strip() else q.stderr.strip()}


def stats(ts):
    return {"median_ms": statistics.median(ts), "min_ms": min(ts), "max_ms": max(ts), "reps": len(ts)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--loop-reps", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_blob_verify_batches_bench_b200.jsonl"))
    a = ap.parse_args()
    lw.set_option("mode", 2)
    lw.set_option("window_bits", 8)
    s = lw.load_trusted_setup_file(os.path.join(ROOT, "tests", "golden", "trusted_setup.txt"))
    lib = lw.load_library()
    sp = lw.api._sp(s)
    recs = [{"kind": "card", **card(), "mode": 2, "window_bits": 8}]

    nmax = max(k * n for k, n in SHAPES)
    d_blobs = torch.empty(nmax * BLOB, dtype=torch.uint8, device="cuda")
    d_com = torch.empty(nmax * 48, dtype=torch.uint8, device="cuda")
    d_pi = torch.empty(nmax * 48, dtype=torch.uint8, device="cuda")
    d_st = torch.zeros(nmax, dtype=torch.int32, device="cuda")
    assert lib.lwkzg_synth_blobs_device(d_blobs.data_ptr(), 0, nmax, None) == 0
    assert lib.lwkzg_commit_and_prove_batch_device(d_com.data_ptr(), d_pi.data_ptr(), d_blobs.data_ptr(), nmax, sp, None, d_st.data_ptr()) == 0
    torch.cuda.synchronize()
    assert d_st.sum().item() == 0
    h_blobs, h_com, h_pi = (t.cpu().pin_memory() for t in (d_blobs, d_com, d_pi))
    d_ok = torch.zeros(nmax, dtype=torch.int32, device="cuda")
    d_bst = torch.zeros(nmax, dtype=torch.int32, device="cuda")
    h_ok = (ctypes.c_bool * nmax)()
    h_bst = (ctypes.c_int * nmax)()

    def sync_ms(fn):
        torch.cuda.synchronize()
        t = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t) * 1e3

    for k, nb in SHAPES:
        offsets = (ctypes.c_uint64 * (k + 1))(*[nb * i for i in range(k + 1)])

        def new_device():
            rc = lib.lwkzg_verify_blob_kzg_proof_batches_device(d_ok.data_ptr(), d_blobs.data_ptr(), d_com.data_ptr(), d_pi.data_ptr(), offsets, k, sp,
                                                                None, d_bst.data_ptr())
            assert rc == 0, lw.last_error()

        def new_device_ms():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            new_device()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1)

        def new_pinned():
            rc = lib.lwkzg_verify_blob_kzg_proof_batches(h_ok, h_blobs.data_ptr(), h_com.data_ptr(), h_pi.data_ptr(), offsets, k, sp, h_bst)
            assert rc == 0, lw.last_error()

        loop_ok = []

        def loop_device():
            loop_ok.clear()
            for b in range(k):
                loop_ok.append(lw.verify_blob_kzg_proof_batch_device(d_blobs.data_ptr() + b * nb * BLOB, d_com.data_ptr() + b * nb * 48,
                                                                     d_pi.data_ptr() + b * nb * 48, nb, s))

        def loop_pinned():
            loop_ok.clear()
            for b in range(k):
                loop_ok.append(lw.verify_blob_kzg_proof_batch_ptr(h_blobs.data_ptr() + b * nb * BLOB, h_com.data_ptr() + b * nb * 48,
                                                                  h_pi.data_ptr() + b * nb * 48, nb, s))

        new_device_ms()
        sync_ms(new_pinned)
        td = [new_device_ms() for _ in range(a.reps)]
        assert d_ok[:k].cpu().tolist() == [1] * k and d_bst[:k].cpu().tolist() == [0] * k
        th = [sync_ms(new_pinned) for _ in range(a.reps)]
        assert all(h_ok[i] for i in range(k)) and all(h_bst[i] == 0 for i in range(k))
        lreps = a.reps if k <= 256 else a.loop_reps
        sync_ms(loop_device if k <= 256 else (lambda: None))
        tld = [sync_ms(loop_device) for _ in range(lreps)]
        assert loop_ok == [True] * k
        tlp = [sync_ms(loop_pinned) for _ in range(lreps)]
        assert loop_ok == [True] * k
        rec = {"kind": "shape", "K": k, "n_b": nb, "blobs": k * nb, "new_device": stats(td), "new_pinned": stats(th), "loop_device": stats(tld),
               "loop_pinned": stats(tlp)}
        rec["speedup_device"] = statistics.median(tld) / statistics.median(td)
        rec["speedup_pinned"] = statistics.median(tlp) / statistics.median(th)
        recs.append(rec)
        print(json.dumps(rec), flush=True)

    # per-stage kernel times of the new call at 128 x 6, device-resident, from the profiler
    from torch.profiler import ProfilerActivity, profile

    k, nb = SHAPES[0]
    offsets = (ctypes.c_uint64 * (k + 1))(*[nb * i for i in range(k + 1)])
    call = lambda: lib.lwkzg_verify_blob_kzg_proof_batches_device(d_ok.data_ptr(), d_blobs.data_ptr(), d_com.data_ptr(), d_pi.data_ptr(),  # noqa: E731
                                                                  offsets, k, sp, None, d_bst.data_ptr())
    call()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call()
        torch.cuda.synchronize()
    kern = {}
    for e in prof.key_averages():
        kern[e.key.split("(")[0]] = getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0)) / 1e3   # ms
    stages = {name: sum(v for kk, v in kern.items() if any(f in kk for f in frags)) for name, frags in STAGES.items()}
    rec = {"kind": "stages", "K": k, "n_b": nb, "stage_kernel_ms": stages, "kernel_ms": kern}
    recs.append(rec)
    print(json.dumps(rec), flush=True)
    s.free()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for r in recs:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
