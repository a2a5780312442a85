#!/usr/bin/env python3
"""Cell-proof verification straight from blobs (lwkzg_verify_blob_cell_kzg_proof_batches[_device]) in the shape a
mempool meets it: MODE_DENEB, synthetic blobs, one batch per blob transaction (its blobs, one commitment per blob, 128
cell proofs per blob).

For each T x B shape (T transactions of B blobs): the device form (CUDA events, after a warm-up call) and the host
form from pinned memory, against the composition the call replaces, timed the same way:
  - device: lwkzg_compute_cells_and_kzg_proofs_batch_device (cells only), the replicated commitments and the cell
    indices built on the device, lwkzg_verify_cell_kzg_proof_batches_device;
  - host: lwkzg_compute_cells_and_kzg_proofs_batch (cells only, into pinned memory), the replicated commitments and
    the cell indices built on the host, lwkzg_verify_cell_kzg_proof_batches from pinned memory.
Every verdict and status of every timed call is checked.  Then, in a separate profiled call per shape (torch.profiler
with CUDA activities), the kernel time of each stage of the new device form: extension, decode (blob check, point
decompression, cell parsing, broadcast), dedup, hash, scalars, MSM, pairing.  Card name and power limit are read in
the same run.

python tools/blob_cell_verify_bench.py [--shapes 1x1,1x6,64x6,128x6,888x1] [--out FILE]"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import lambdaworks_kzg_b200 as lw  # noqa: E402

STAGES = [("cell_poly", "extension"), ("le_blob_check", "decode"), ("g1_decompress", "decode"), ("cell_parse", "decode"),
          ("cell_blob_broadcast", "decode"), ("cell_batches_prepare", "dedup"), ("cell_batches_challenge", "hash"), ("cell_interp", "scalars"),
          ("cell_batches_finish", "scalars"), ("cell_segmsm", "msm"), ("batch_final", "pairing"), ("cell_batches_fold", "fold")]


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def event_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def wall_ms(fn, reps):
    fn()
    t = time.perf_counter()
    for _ in range(reps):
        fn()
    return (time.perf_counter() - t) / reps * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="1x1,1x6,64x6,128x6,888x1")
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
    nb_max = max(t * b for t, b in shapes)
    blobs = b"".join(lw.synth_blob_host(k) for k in range(nb_max))
    coms, st = lw.blob_to_kzg_commitment_batch(blobs, nb_max, s)
    _, proofs, st2 = lw.compute_cells_and_kzg_proofs_batch(blobs, nb_max, s, want_cells=False)
    assert st == [0] * nb_max and st2 == [0] * nb_max
    lib = lw.load_library()

    for T, B in shapes:
        n = T * B
        offs = [t * B for t in range(T + 1)]
        offsets = (ctypes.c_uint64 * (T + 1))(*offs)
        cell_offsets = (ctypes.c_uint64 * (T + 1))(*[o * 128 for o in offs])
        h_blob = torch.frombuffer(bytearray(blobs[: n * 131072]), dtype=torch.uint8).pin_memory()
        h_com = torch.frombuffer(bytearray(b"".join(coms[:n])), dtype=torch.uint8).pin_memory()
        h_prf = torch.frombuffer(bytearray(proofs[: n * 128 * 48]), dtype=torch.uint8).pin_memory()
        d_blob, d_com, d_prf = h_blob.cuda(), h_com.cuda(), h_prf.cuda()
        d_ok = torch.full((T,), -1, dtype=torch.int32, device="cuda")
        d_st = torch.full((T,), -1, dtype=torch.int32, device="cuda")
        reps = max(3, min(20, 768 // n))

        def check_dev():
            assert d_ok.tolist() == [1] * T and d_st.tolist() == [0] * T, "device verdicts"
            d_ok.fill_(-1)
            d_st.fill_(-1)

        # the new call, device form
        def dev_call():
            assert lib.lwkzg_verify_blob_cell_kzg_proof_batches_device(d_ok.data_ptr(), d_blob.data_ptr(), d_com.data_ptr(), d_prf.data_ptr(), offsets, T,
                                                                       s.ptr, stream, d_st.data_ptr()) == 0

        dev_ms = event_ms(dev_call, reps)
        check_dev()
        # the composition it replaces, device form: cells, replicated commitments and indices, the cell batches call
        d_cells = torch.empty((n * 128 * 2048,), dtype=torch.uint8, device="cuda")
        d_cst = torch.empty((n,), dtype=torch.int32, device="cuda")
        d_ar = torch.arange(128, dtype=torch.int64, device="cuda")

        def comp_dev_call():
            assert lib.lwkzg_compute_cells_and_kzg_proofs_batch_device(d_cells.data_ptr(), None, d_blob.data_ptr(), n, s.ptr, stream, d_cst.data_ptr()) == 0
            d_rep = d_com.view(n, 48).repeat_interleave(128, dim=0)
            d_idx = d_ar.repeat(n)
            assert lib.lwkzg_verify_cell_kzg_proof_batches_device(d_ok.data_ptr(), d_rep.data_ptr(), d_idx.data_ptr(), d_cells.data_ptr(), d_prf.data_ptr(),
                                                                  cell_offsets, T, s.ptr, stream, d_st.data_ptr()) == 0

        comp_dev_ms = event_ms(comp_dev_call, reps)
        assert d_cst.tolist() == [0] * n
        check_dev()
        # the new call, host form from pinned memory
        oks = (ctypes.c_bool * T)()
        hst = (ctypes.c_int * T)()

        def host_call():
            assert lib.lwkzg_verify_blob_cell_kzg_proof_batches(oks, h_blob.data_ptr(), h_com.data_ptr(), h_prf.data_ptr(), offsets, T, s.ptr, hst) == 0

        hreps = max(2, reps // 2)
        host_ms = wall_ms(host_call, hreps)
        assert list(oks) == [True] * T and list(hst) == [0] * T, "host verdicts"
        # the composition, host form: cells into pinned memory, the arrays built by the caller, the cell batches call
        h_cells = torch.empty((n * 128 * 2048,), dtype=torch.uint8).pin_memory()
        h_cst = (ctypes.c_int * n)()
        h_com_np = h_com.numpy().reshape(n, 48)
        h_rep = torch.empty((n * 128 * 48,), dtype=torch.uint8).pin_memory()
        h_idx = torch.empty((n * 128,), dtype=torch.int64).pin_memory()
        oks2 = (ctypes.c_bool * T)()
        hst2 = (ctypes.c_int * T)()

        def comp_host_call():
            assert lib.lwkzg_compute_cells_and_kzg_proofs_batch(h_cells.data_ptr(), None, h_blob.data_ptr(), n, s.ptr, h_cst) == 0
            h_rep.numpy()[:] = np.repeat(h_com_np, 128, axis=0).reshape(-1)
            h_idx.numpy()[:] = np.tile(np.arange(128, dtype=np.int64), n)
            assert lib.lwkzg_verify_cell_kzg_proof_batches(oks2, h_rep.data_ptr(), h_idx.data_ptr(), h_cells.data_ptr(), h_prf.data_ptr(), cell_offsets, T,
                                                           s.ptr, hst2) == 0

        comp_host_ms = wall_ms(comp_host_call, hreps)
        assert list(h_cst) == [0] * n and list(oks2) == [True] * T and list(hst2) == [0] * T, "composed host verdicts"
        # kernel time per stage of one device call of the new form, profiled on its own
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            dev_call()
            torch.cuda.synchronize()
        check_dev()
        stage_us = {}
        for ev in prof.key_averages():
            stg = next((v for k, v in STAGES if k in ev.key), None)
            if stg:
                stage_us[stg] = stage_us.get(stg, 0.0) + ev.device_time_total
        emit({"T": T, "B": B, "blobs": n, "cells": n * 128, "device_ms": round(dev_ms, 3), "composed_device_ms": round(comp_dev_ms, 3),
              "host_pinned_ms": round(host_ms, 3), "composed_host_pinned_ms": round(comp_host_ms, 3),
              "speedup_device": round(comp_dev_ms / dev_ms, 2), "speedup_host": round(comp_host_ms / host_ms, 2),
              "stage_kernel_ms": {k: round(v / 1e3, 3) for k, v in sorted(stage_us.items())}, "reps": reps, "host_reps": hreps, "verdicts_checked": True})
        del d_blob, d_com, d_prf, d_cells, h_blob, h_com, h_prf, h_cells, h_rep, h_idx
        torch.cuda.empty_cache()
    s.free()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
