#!/usr/bin/env python3
"""Many cell-proof batches per call (lwkzg_verify_cell_kzg_proof_batches[_device]) in the shape a PeerDAS node meets
them: MODE_DENEB, synthetic blobs, one batch per data column sidecar (the cells and proofs of B blobs at one column).

For each K x B shape: device-resident time (CUDA events, after a warm-up call), the host API from pinned memory, and
the loop of K single verify_cell_kzg_proof_batch calls from the same process.  1 x 1776 is one batch of 1776 cells (48
blobs x 37 columns).  Every verdict and status is checked.  Then, in a separate profiled call per shape (torch.profiler
with CUDA activities), the kernel time of each stage of the device form: decode (cell parsing + point decompression),
dedup, hash, scalars, MSM, pairing.  Card name and power limit are read in the same run.

python tools/cell_verify_bench.py [--shapes 128x6,128x48,32x48,8x48,1x128,1x1776] [--out FILE]"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import lambdaworks_kzg_b200 as lw  # noqa: E402

NBLOBS = 48
STAGES = [("cell_parse", "decode"), ("g1_decompress", "decode"), ("cell_batches_prepare", "dedup"), ("cell_batches_challenge", "hash"),
          ("cell_interp", "scalars"), ("cell_batches_finish", "scalars"), ("cell_segmsm", "msm"), ("batch_final", "pairing"),
          ("cell_batches_fold", "fold")]


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="128x6,128x48,32x48,8x48,1x128,1x1776")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    shapes = [tuple(int(v) for v in x.split("x")) for x in a.shapes.split(",")]
    lines = []

    def emit(d):
        lines.append(json.dumps(d))
        print(lines[-1], flush=True)

    emit({"card": card(), "cell_chunk_blobs": lw.get_option("cell_chunk_blobs")})
    lw.set_option("mode", 2)
    lw.set_option("window_bits", 8)
    s = lw.load_trusted_setup_file(os.path.join(ROOT, "tests", "golden", "trusted_setup.txt"))
    lw.set_option("mode", 0)
    torch.cuda.set_device(0)
    stream = torch.cuda.current_stream().cuda_stream
    nb_max = max([b for k, b in shapes if b != 1776] + [NBLOBS])
    blobs = b"".join(lw.synth_blob_host(k) for k in range(nb_max))
    coms, st = lw.blob_to_kzg_commitment_batch(blobs, nb_max, s)
    cells, proofs, st2 = lw.compute_cells_and_kzg_proofs_batch(blobs, nb_max, s)
    assert st == [0] * nb_max and st2 == [0] * nb_max
    lib = lw.load_library()

    for K, B in shapes:
        # (blob, column) of every cell, batch-major
        if B == 1776:
            sel = [[(b, c) for b in range(NBLOBS) for c in range(37)]]
        elif K == 1:
            sel = [[(b % nb_max, (b // nb_max) % 128) for b in range(B)]]
        else:
            sel = [[(b, col) for b in range(B)] for col in range(K)]
        offs = [0]
        for x in sel:
            offs.append(offs[-1] + len(x))
        flat = [p for x in sel for p in x]
        n = len(flat)
        com = b"".join(coms[b] for b, _ in flat)
        idx = [c for _, c in flat]
        cel = b"".join(cells[(b * 128 + c) * 2048: (b * 128 + c + 1) * 2048] for b, c in flat)
        prf = b"".join(proofs[(b * 128 + c) * 48: (b * 128 + c + 1) * 48] for b, c in flat)
        h_com, h_cel, h_prf = (torch.frombuffer(bytearray(x), dtype=torch.uint8).pin_memory() for x in (com, cel, prf))
        h_idx = torch.tensor(idx, dtype=torch.int64).pin_memory()
        d_com, d_cel, d_prf, d_idx = h_com.cuda(), h_cel.cuda(), h_prf.cuda(), h_idx.cuda()
        d_ok = torch.full((K,), -1, dtype=torch.int32, device="cuda")
        d_st = torch.full((K,), -1, dtype=torch.int32, device="cuda")
        offsets = (ctypes.c_uint64 * (K + 1))(*offs)
        reps = max(3, min(20, 2048 // n))

        def dev_call():
            assert lib.lwkzg_verify_cell_kzg_proof_batches_device(d_ok.data_ptr(), d_com.data_ptr(), d_idx.data_ptr(), d_cel.data_ptr(), d_prf.data_ptr(),
                                                                  offsets, K, s.ptr, stream, d_st.data_ptr()) == 0

        dev_call()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            dev_call()
        e1.record()
        torch.cuda.synchronize()
        dev_ms = e0.elapsed_time(e1) / reps
        assert d_ok.tolist() == [1] * K and d_st.tolist() == [0] * K, "device verdicts"
        # host API from pinned memory
        oks = (ctypes.c_bool * K)()
        hst = (ctypes.c_int * K)()
        host_call = lambda: lib.lwkzg_verify_cell_kzg_proof_batches(oks, h_com.data_ptr(), h_idx.data_ptr(), h_cel.data_ptr(), h_prf.data_ptr(),  # noqa: E731
                                                                    offsets, K, s.ptr, hst)
        assert host_call() == 0
        hreps = max(2, reps // 2)
        t = time.perf_counter()
        for _ in range(hreps):
            assert host_call() == 0
        host_ms = (time.perf_counter() - t) / hreps * 1e3
        assert list(oks) == [True] * K and list(hst) == [0] * K, "host verdicts"
        # the loop of K single calls (inputs prepared beforehand; one full loop, after one warm-up call)
        singles = []
        for b in range(K):
            o0, o1 = offs[b], offs[b + 1]
            singles.append((com[o0 * 48: o1 * 48], (ctypes.c_uint64 * (o1 - o0))(*idx[o0:o1]), cel[o0 * 2048: o1 * 2048], prf[o0 * 48: o1 * 48], o1 - o0))
        ok1 = ctypes.c_bool(False)
        assert lib.verify_cell_kzg_proof_batch(ctypes.byref(ok1), *singles[0], s.ptr) == 0 and ok1.value
        t = time.perf_counter()
        for args in singles:
            ok1 = ctypes.c_bool(False)
            assert lib.verify_cell_kzg_proof_batch(ctypes.byref(ok1), *args, s.ptr) == 0 and ok1.value
        loop_ms = (time.perf_counter() - t) * 1e3
        # kernel time per stage of one device call, profiled on its own
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            dev_call()
            torch.cuda.synchronize()
        stage_us = {}
        for ev in prof.key_averages():
            st = next((v for k, v in STAGES if k in ev.key), None)
            if st:
                stage_us[st] = stage_us.get(st, 0.0) + ev.device_time_total
        emit({"K": K, "B": B, "cells": n, "device_ms": round(dev_ms, 3), "host_pinned_ms": round(host_ms, 3), "single_call_loop_ms": round(loop_ms, 2),
              "stage_kernel_ms": {k: round(v / 1e3, 3) for k, v in sorted(stage_us.items())},
              "single_call_loops": 1, "speedup_device_vs_loop": round(loop_ms / dev_ms, 1), "speedup_host_vs_loop": round(loop_ms / host_ms, 1),
              "reps": reps, "verdicts_checked": True})
        del d_com, d_cel, d_prf, d_idx, h_com, h_cel, h_prf
    s.free()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
