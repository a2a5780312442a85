"""Load time of a c-kzg-4844 trusted setup (lwkzg_load_trusted_setup_file_ckzg) against the reference-format loader
(load_trusted_setup_file) on the same tau, MODE_DENEB, at window_bits 8 and 16: the median of 3 loads each, total
(host clock) and per phase (lwkzg_last_load_times: decode and setup check by CUDA events, Lagrange conversion and
context build by host clock).  The tau = 1337 golden setup stands in for the mainnet file; both have 4096 + 65 points.

    python tools/ckzg_setup_bench.py [--out profiles/r03_ckzg_setup_load_b200.jsonl]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import lambdaworks_kzg_b200 as lw  # noqa: E402
from tests._ckzg_setup import golden_sections, lagrange_from_settings, write_text  # noqa: E402

SETUP = os.path.join(ROOT, "tests", "golden", "trusted_setup.txt")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    name, power = [x.strip() for x in q.stdout.strip().split(",")[:2]]
    return name, power


def timed(load):
    t0 = time.perf_counter()
    s = load()
    total = (time.perf_counter() - t0) * 1e3
    phases = lw.last_load_times()
    s.free()
    return dict(total_ms=total, **phases)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_ckzg_setup_load_b200.jsonl"))
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    lw.load_library()
    name, power = card()
    lw.set_option("window_bits", 8)
    lw.set_option("mode", 1)
    mono, g2 = golden_sections()
    s = lw.load_trusted_setup(b"".join(mono), b"".join(g2))
    lag = lagrange_from_settings(s)
    s.free()
    lw.set_option("mode", 2)
    with tempfile.NamedTemporaryFile(suffix=".txt", delete=False) as f:
        f.write(write_text(lag, g2, mono))
        ckzg_path = f.name
    rows = []
    try:
        for wb in (8, 16):
            lw.set_option("window_bits", wb)
            loaders = {"load_trusted_setup_file": lambda: lw.load_trusted_setup_file(SETUP),
                       "lwkzg_load_trusted_setup_file_ckzg": lambda: lw.load_trusted_setup_file_ckzg(ckzg_path)}
            runs = {k: [] for k in loaders}
            timed(loaders["load_trusted_setup_file"])   # warm-up: module load, first allocations
            for _ in range(a.reps):   # alternate the two loaders
                for k, fn in loaders.items():
                    runs[k].append(timed(fn))
            for k, rs in runs.items():
                row = {"loader": k, "mode": 2, "window_bits": wb, "reps": a.reps, "gpu": name, "power_limit": power}
                for f in ("total_ms", "decode_ms", "check_ms", "convert_ms", "build_ms"):
                    row[f + "_median"] = round(statistics.median(r[f] for r in rs), 3)
                row["total_ms_all"] = [round(r["total_ms"], 3) for r in rs]
                rows.append(row)
                print(json.dumps(row), flush=True)
    finally:
        os.unlink(ckzg_path)
        lw.set_option("mode", 0)
        lw.set_option("window_bits", 16)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
