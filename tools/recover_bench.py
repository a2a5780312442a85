#!/usr/bin/env python3
"""Batched cell recovery (lwkzg_recover_cells_and_kzg_proofs_batch[_device]) in the shape a PeerDAS node meets it:
MODE_DENEB, synthetic blobs, the same 64 of the 128 columns kept for every blob of a block.

For each n: device-resident time (CUDA events, after a warm-up call), the host API from pinned memory, and the single
recover_cells_and_kzg_proofs call from the same process.  Every output is checked, outside the timed regions, against
lwkzg_compute_cells_and_kzg_proofs_batch on the original blobs.  Card name and power limit are read in the same run.

python tools/recover_bench.py [--sizes 1,16,64,128,256,888] [--out FILE]"""
import argparse
import ctypes
import json
import os
import random
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import lambdaworks_kzg_b200 as lw  # noqa: E402

CB, PB = 128 * 2048, 128 * 48


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1,16,64,128,256,888")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    sizes = [int(x) for x in a.sizes.split(",")]
    nmax = max(sizes)
    lines = []

    def emit(d):
        lines.append(json.dumps(d))
        print(lines[-1], flush=True)

    emit({"card": card(), "cell_chunk_blobs": lw.get_option("cell_chunk_blobs")})
    lw.set_option("mode", 2)
    lw.set_option("window_bits", 8)   # the commitment table is not used here; the FK20 table keeps its default window
    s = lw.load_trusted_setup_file(os.path.join(ROOT, "tests", "golden", "trusted_setup.txt"))
    lw.set_option("mode", 0)
    torch.cuda.set_device(0)
    stream = torch.cuda.current_stream().cuda_stream
    keep = sorted(random.Random(7594).sample(range(128), 64))

    # originals and their cells / proofs through the compute batch (host API)
    blobs = b"".join(lw.synth_blob_host(k) for k in range(nmax))
    want_c, want_p, st = lw.compute_cells_and_kzg_proofs_batch(blobs, nmax, s)
    assert st == [0] * nmax
    emit({"cell_window_bits": lw.cell_window_bits(s), "kept_columns": keep})
    all_cells = torch.frombuffer(bytearray(want_c), dtype=torch.uint8).view(nmax, 128, 2048)
    kept = all_cells[:, keep, :].contiguous()                    # nmax x 64 x 2048
    idx = torch.tensor(keep, dtype=torch.int64).repeat(nmax)      # nmax x 64 (same bytes as uint64)
    d_in, d_idx = kept.cuda().view(-1), idx.cuda()
    h_in, h_idx = kept.view(-1).pin_memory(), idx.pin_memory()
    lib = lw.load_library()

    # the single call, blob 0
    one = [bytes(kept[0, j].numpy()) for j in range(64)]
    lw.recover_cells_and_kzg_proofs(keep, one, s)
    reps1 = 10
    t = time.perf_counter()
    for _ in range(reps1):
        rc, rp = lw.recover_cells_and_kzg_proofs(keep, one, s)
    single_ms = (time.perf_counter() - t) / reps1 * 1e3
    assert b"".join(rc) == want_c[:CB] and b"".join(rp) == want_p[:PB]
    emit({"single_call_ms": round(single_ms, 3), "reps": reps1})

    for n in sizes:
        d_c = torch.zeros(n * CB, dtype=torch.uint8, device="cuda")
        d_p = torch.zeros(n * PB, dtype=torch.uint8, device="cuda")
        d_st = torch.full((n,), -1, dtype=torch.int32, device="cuda")
        reps = max(3, min(20, 512 // n))

        def dev_call():
            lw.recover_cells_and_kzg_proofs_batch_device(d_c.data_ptr(), d_p.data_ptr(), d_idx.data_ptr(), d_in.data_ptr(), 64, n, s, stream,
                                                         d_st.data_ptr())

        dev_call()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            dev_call()
        e1.record()
        torch.cuda.synchronize()
        dev_ms = e0.elapsed_time(e1) / reps
        assert d_st.tolist() == [0] * n
        assert bytes(d_c.cpu().numpy()) == want_c[: n * CB] and bytes(d_p.cpu().numpy()) == want_p[: n * PB], "device outputs differ"
        # host API, pinned buffers
        hc = torch.zeros(n * CB, dtype=torch.uint8).pin_memory()
        hp = torch.zeros(n * PB, dtype=torch.uint8).pin_memory()
        hst = (ctypes.c_int * n)()
        host_call = lambda: lib.lwkzg_recover_cells_and_kzg_proofs_batch(hc.data_ptr(), hp.data_ptr(), h_idx.data_ptr(), h_in.data_ptr(), 64, n,  # noqa: E731
                                                                         s.ptr, hst)
        assert host_call() == 0
        hreps = max(2, reps // 2)
        t = time.perf_counter()
        for _ in range(hreps):
            assert host_call() == 0
        host_ms = (time.perf_counter() - t) / hreps * 1e3
        assert list(hst) == [0] * n
        assert bytes(hc.numpy()) == want_c[: n * CB] and bytes(hp.numpy()) == want_p[: n * PB], "host outputs differ"
        emit({"n": n, "device_ms": round(dev_ms, 3), "device_ms_per_blob": round(dev_ms / n, 4), "host_pinned_ms": round(host_ms, 3),
              "host_pinned_ms_per_blob": round(host_ms / n, 4), "n_single_calls_ms": round(n * single_ms, 1),
              "speedup_vs_single_calls": round(n * single_ms / host_ms, 1), "reps": reps, "outputs_checked": True})
        del d_c, d_p, hc, hp
    s.free()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
