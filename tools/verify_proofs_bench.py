#!/usr/bin/env python3
"""Many single-opening checks per call, lwkzg_verify_kzg_proofs[_device], against n calls of verify_kzg_proof.

MODE_DENEB, the test setup's tables at window 8 (the call uses no fixed-base table), 64 distinct valid openings tiled
to n.  For each n: verdicts per second device-resident (CUDA events around each call) and from pinned host memory
(host clock around each synchronous call), median and spread of --reps repetitions after a warm-up; for n <= 256 the
median time of one verify_kzg_proof call, times n, next to it.  The verdicts are checked against the known answer
(all true) on every timed size.  A profiler run at the largest n gives the pairing kernel's time alone, and with the
MAC32 work model below and lwkzg_imad_peak from the same run its share of the multiplier's peak.  Card name and
power limit are read in the same run.

python tools/verify_proofs_bench.py [--sizes 1,32,1024,16384,131072] [--reps 7] [--out FILE]"""
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

R = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001

# Work model, in 32-bit multiply-accumulates (MAC32) per item.  A Montgomery product of two 12-limb Fp elements is
# 2 x 144 MAC32.  Fp products per item, counted from the code:
#   Miller loop: 63 Fp12 squarings (2 Fp6 products = 36 Fp) + 2 x 68 sparse line products (13 Fp2 products + 2 = 41 Fp)
#   final exponentiation: 5 x pow_x (63 cyclotomic squarings of 18 Fp + 5 Fp12 products of 54 Fp) + ~15 Fp12
#     products and Frobenius maps (~800 Fp)
#   G1 stage: 128 doublings (9 Fp) + 128 table additions (14 Fp) + 15 table-building additions (10 Fp) + one inversion
#     (~60 Fp equivalents)
#   decoding: two square roots (~450 Fp each) and two r-torsion tests (~1200 Fp each)
FP_MAC32 = 2 * 144
FP_PAIRING = 63 * 36 + 136 * 41 + 5 * (63 * 18 + 5 * 54) + 800
FP_G1 = 128 * 9 + 128 * 14 + 15 * 10 + 60
FP_DECODE = 2 * (450 + 1200)
MODEL = {"pairing_mac32": FP_PAIRING * FP_MAC32, "g1_stage_mac32": FP_G1 * FP_MAC32, "decode_mac32": FP_DECODE * FP_MAC32}
MODEL["total_mac32"] = sum(MODEL.values())


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[-1] if q.stdout.strip() else q.stderr.strip()}


def stats(ts):
    return {"median_ms": statistics.median(ts), "min_ms": min(ts), "max_ms": max(ts)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1,32,1024,16384,131072")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_verify_proofs_bench_b200.jsonl"))
    a = ap.parse_args()
    sizes = [int(x) for x in a.sizes.split(",")]
    lw.set_option("mode", 2)
    lw.set_option("window_bits", 8)
    s = lw.load_trusted_setup_file(os.path.join(ROOT, "tests", "golden", "trusted_setup.txt"))
    lib = lw.load_library()
    sp = lw.api._sp(s)
    recs = [{"kind": "card", **card(), "model_per_item": MODEL}]

    m = 64
    blobs = b"".join(lw.synth_blob_host(k) for k in range(m))
    zs = [((k * 0x9E3779B97F4A7C15) ** 3 % R).to_bytes(32, "big") for k in range(m)]
    coms, st = lw.blob_to_kzg_commitment_batch(blobs, m, s)
    proofs, ys, st2 = lw.compute_kzg_proof_batch(blobs, b"".join(zs), m, s)
    assert st == [0] * m and st2 == [0] * m
    base = [b"".join(coms), b"".join(zs), b"".join(ys), b"".join(proofs)]
    nmax = max(sizes)
    tiles = (nmax + m - 1) // m
    host = [torch.frombuffer(bytearray(b * tiles), dtype=torch.uint8)[: nmax * (len(b) // m)].pin_memory() for b in base]
    dev = [h.cuda() for h in host]
    d_ok = torch.zeros(nmax, dtype=torch.int32, device="cuda")
    d_st = torch.zeros(nmax, dtype=torch.int32, device="cuda")
    h_ok = (ctypes.c_bool * nmax)()
    h_st = (ctypes.c_int * nmax)()

    def run_dev(n):
        rc = lib.lwkzg_verify_kzg_proofs_device(d_ok.data_ptr(), dev[0].data_ptr(), dev[1].data_ptr(), dev[2].data_ptr(), dev[3].data_ptr(), n, sp,
                                                None, d_st.data_ptr())
        assert rc == 0, lw.last_error()

    def run_host(n):
        rc = lib.lwkzg_verify_kzg_proofs(h_ok, host[0].data_ptr(), host[1].data_ptr(), host[2].data_ptr(), host[3].data_ptr(), n, sp, h_st)
        assert rc == 0, lw.last_error()

    def dev_ms(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        run_dev(n)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    def host_ms(n):
        t = time.perf_counter()
        run_host(n)
        return (time.perf_counter() - t) * 1e3

    single = None
    for n in sizes:
        dev_ms(n)
        host_ms(n)
        td = [dev_ms(n) for _ in range(a.reps)]
        th = [host_ms(n) for _ in range(a.reps)]
        assert d_ok[:n].cpu().tolist() == [1] * n and d_st[:n].cpu().tolist() == [0] * n
        assert all(h_ok[i] for i in range(n)) and all(h_st[i] == 0 for i in range(n))
        rec = {"kind": "size", "n": n, "device": stats(td), "pinned_host": stats(th),
               "device_verdicts_per_s": n / (statistics.median(td) * 1e-3), "pinned_host_verdicts_per_s": n / (statistics.median(th) * 1e-3)}
        if n <= 256:
            if single is None:
                it = (coms[0], zs[0], ys[0], proofs[0])
                assert lw.verify_kzg_proof(*it, s)
                ts = []
                for _ in range(max(a.reps, 15)):
                    t = time.perf_counter()
                    lw.verify_kzg_proof(*it, s)
                    ts.append((time.perf_counter() - t) * 1e3)
                single = statistics.median(ts)
            rec["single_call_median_ms"] = single
            rec["n_single_calls_ms"] = n * single
        recs.append(rec)
        print(json.dumps(rec), flush=True)

    # the pairing kernel alone, from the profiler, at the largest n; the multiplier's peak from the same run
    peak = lw.imad_peak(0)
    from torch.profiler import ProfilerActivity, profile

    run_dev(nmax)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run_dev(nmax)
        torch.cuda.synchronize()
    kern = {}
    for e in prof.key_averages():
        if "verify_proofs" in e.key or "decompress" in e.key:
            kern[e.key.split("(")[0]] = getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0)) / 1e3   # ms
    pair_ms = sum(v for k, v in kern.items() if "pairing" in k)
    rec = {"kind": "kernels", "n": nmax, "kernel_ms": kern, "imad_peak_mac32_per_s": peak,
           "pairing_share_of_imad_peak": (MODEL["pairing_mac32"] * nmax / (pair_ms * 1e-3)) / peak if pair_ms and peak else None,
           "model_ceiling_verdicts_per_s": peak / MODEL["total_mac32"] if peak else None}
    recs.append(rec)
    print(json.dumps(rec), flush=True)

    # the A/B of the pairing stage's two layouts (thread per item against a 64-lane group per item) was measured while
    # both were built, and decided the layout; the other one is deleted, its records are kept
    if os.path.exists(a.out):
        recs += [json.loads(ln) for ln in open(a.out) if ln.strip() and json.loads(ln).get("kind") == "pairing_layout_ab"]
    s.free()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        for r in recs:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
