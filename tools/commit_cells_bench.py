#!/usr/bin/env python3
"""Commitments, cell proofs and (optionally) cells in one call, lwkzg_commit_and_compute_cells_and_kzg_proofs_batch[_device],
against the composition it replaces: lwkzg_blob_to_kzg_commitment_batch[_device] followed by
lwkzg_compute_cells_and_kzg_proofs_batch[_device] on the same blobs.

MODE_DENEB, the default tables (fixed-base window 16 = 100 GiB commitment table, cell window 13 = 29 GiB FK20 table),
synthetic blobs.  For each n: the device-resident form (CUDA events around each call) and the host form from pinned
memory (host clock around each synchronous call), each without and with cells.  Every pair is timed A/B, alternating
which goes first, 10 repetitions after a warm-up of both; the median and the spread (min, max) of each are reported.
The bytes of both sides are compared once per n and form.  Card name and power limit are read in the same run, and the
free HBM after the largest pass is recorded.

python tools/commit_cells_bench.py [--sizes 1,6,128,888,1776] [--reps 10] [--out FILE]"""
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

CELL, PROOFS = 128 * 2048, 128 * 48


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[-1] if q.stdout.strip() else q.stderr.strip()}


def device_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def host_ms(fn):
    t = time.perf_counter()
    fn()
    return (time.perf_counter() - t) * 1e3


def ab(timer, fa, fb, reps):
    """A/B timing, alternating which runs first; -> (times of a, times of b)"""
    timer(fa)
    timer(fb)
    ta, tb = [], []
    for r in range(reps):
        if r % 2 == 0:
            ta.append(timer(fa))
            tb.append(timer(fb))
        else:
            tb.append(timer(fb))
            ta.append(timer(fa))
    return ta, tb


def summary(ts):
    return {"median_ms": round(statistics.median(ts), 3), "min_ms": round(min(ts), 3), "max_ms": round(max(ts), 3)}


def load_settings():
    lw.set_option("mode", 2)
    try:
        return lw.load_trusted_setup_file(os.path.join(ROOT, "tests", "golden", "trusted_setup.txt"))
    finally:
        lw.set_option("mode", 0)


class Case:
    """n blobs on the device and in pinned memory, with the output buffers of both sides of each form"""

    def __init__(self, s, n):
        self.s, self.n = s, n
        self.lib = lw.load_library()
        self.stream = torch.cuda.current_stream().cuda_stream
        self.d_blobs = torch.empty((n * 131072,), dtype=torch.uint8, device="cuda")
        lw.synth_blobs_device(self.d_blobs.data_ptr(), 0, n, self.stream)
        self.h_blobs = self.d_blobs.cpu().pin_memory()
        self.d = {k: torch.empty((n * b,), dtype=torch.uint8, device="cuda") for k, b in (("c", 48), ("cells", CELL), ("p", PROOFS), ("c2", 48),
                                                                                         ("cells2", CELL), ("p2", PROOFS))}
        self.d_st = torch.empty((3 * n,), dtype=torch.int32, device="cuda")
        self.h = {k: torch.empty((n * b,), dtype=torch.uint8).pin_memory() for k, b in (("c", 48), ("cells", CELL), ("p", PROOFS), ("c2", 48),
                                                                                        ("cells2", CELL), ("p2", PROOFS))}
        self.h_st = [(ctypes.c_int * n)() for _ in range(3)]

    def _ptr(self, m, k, cells):
        return m[k].data_ptr() if (cells or "cells" not in k) else None

    def new_device(self, cells):
        d, st = self.d, self.d_st.data_ptr()
        assert self.lib.lwkzg_commit_and_compute_cells_and_kzg_proofs_batch_device(d["c"].data_ptr(), self._ptr(d, "cells", cells), d["p"].data_ptr(),
                                                                                   self.d_blobs.data_ptr(), self.n, self.s.ptr, self.stream, st) == 0

    def composed_device(self, cells):
        d, st = self.d, self.d_st.data_ptr() + 4 * self.n
        assert self.lib.lwkzg_blob_to_kzg_commitment_batch_device(d["c2"].data_ptr(), self.d_blobs.data_ptr(), self.n, self.s.ptr, self.stream, st) == 0
        assert self.lib.lwkzg_compute_cells_and_kzg_proofs_batch_device(self._ptr(d, "cells2", cells), d["p2"].data_ptr(), self.d_blobs.data_ptr(), self.n,
                                                                        self.s.ptr, self.stream, st + 4 * self.n) == 0

    def new_host(self, cells):
        h, n = self.h, self.n
        assert self.lib.lwkzg_commit_and_compute_cells_and_kzg_proofs_batch(h["c"].data_ptr(), self._ptr(h, "cells", cells), h["p"].data_ptr(),
                                                                            self.h_blobs.data_ptr(), n, self.s.ptr, self.h_st[0]) == 0

    def composed_host(self, cells):
        h, n = self.h, self.n
        assert self.lib.lwkzg_blob_to_kzg_commitment_batch(h["c2"].data_ptr(), self.h_blobs.data_ptr(), n, self.s.ptr, self.h_st[1]) == 0
        assert self.lib.lwkzg_compute_cells_and_kzg_proofs_batch(self._ptr(h, "cells2", cells), h["p2"].data_ptr(), self.h_blobs.data_ptr(), n, self.s.ptr,
                                                                 self.h_st[2]) == 0

    def check(self, m, cells):
        """both sides wrote the same bytes and every status is 0"""
        if m is self.d:
            torch.cuda.synchronize()
            assert self.d_st.tolist() == [0] * (3 * self.n), "device statuses"
        else:
            assert [list(a) for a in self.h_st] == [[0] * self.n] * 3, "host statuses"
        for a, b in (("c", "c2"), ("p", "p2")) + ((("cells", "cells2"),) if cells else ()):
            assert torch.equal(m[a], m[b]), (a, self.n)
        for t in m.values():
            t.fill_(0x5A)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1,6,128,888,1776")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_commit_cells_bench_b200.jsonl"))
    a = ap.parse_args()
    lines = []

    def emit(d):
        lines.append(json.dumps(d))
        print(lines[-1], flush=True)

    torch.cuda.set_device(0)
    s = load_settings()
    emit({"card": card(), "mode": 2, "window_bits": lw.window_bits(s), "cell_chunk_blobs": lw.get_option("cell_chunk_blobs"),
          "chunk_blobs": lw.get_option("chunk_blobs"), "reps": a.reps})
    for n in [int(x) for x in a.sizes.split(",")]:
        c = Case(s, n)
        for form, m, new, composed, timer in (("device", c.d, c.new_device, c.composed_device, device_ms),
                                              ("pinned", c.h, c.new_host, c.composed_host, host_ms)):
            for cells in (False, True):
                for t in m.values():
                    t.fill_(0x5A)
                new(cells)
                composed(cells)
                c.check(m, cells)
                ta, tb = ab(timer, lambda: new(cells), lambda: composed(cells), a.reps)
                sa, sb = summary(ta), summary(tb)
                emit({"n": n, "form": form, "cells": cells, "new": sa, "composed": sb, "saved_ms": round(sb["median_ms"] - sa["median_ms"], 3),
                      "no_slower_beyond_spread": sa["median_ms"] <= sb["max_ms"], "bytes_equal": True})
        free, total = torch.cuda.mem_get_info()
        emit({"n": n, "cell_window_bits": lw.cell_window_bits(s), "hbm_free_gib_after": round(free / 2**30, 2), "hbm_total_gib": round(total / 2**30, 2)})
        del c
        torch.cuda.empty_cache()
    s.free()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
