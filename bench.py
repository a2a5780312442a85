#!/usr/bin/env python3
"""Benchmark of the EIP-4844 hot path (BASELINE.json metric: blobs/sec commit+proof at 1/2/4/8 B200; G1 MSM
points/sec vs CPU reference).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

One step = one pass of the hot path over one batch: for each of 1024 synthetic blobs per GPU (SURVEY §8d generator),
commitment = blob_to_kzg_commitment(blob) and proof = compute_blob_kzg_proof(blob, commitment), through the library's
batch entry point.  Blob batches shard across GPUs with no collective (weak scaling: every rank processes its own
1024 blobs); the timing itself uses a barrier and a max-reduction.

The JSON line (rank 0):
  value         whole-job blobs/s, blobs resident in HBM (device-pointer C ABI call)
  e2e           the same metric through the host-buffer C ABI call (lwkzg_commit_and_prove_batch), H2D of the blobs and
                D2H of commitments / proofs / status inside the timed region; pinned host memory (the headline) and
                pageable memory (what a c-kzg caller passes) side by side
  parity        a sample of every rank's timed outputs compared with the C restatement oracle OUTSIDE the timed region
  roofline      the dominant kernel (batched fixed-base MSM) alone: SURVEY §8d's algorithmic work / its time against
                the integer-multiply peak, plus the fractions against what the kernel really executes and against this
                algorithm's own minimum; HBM traffic from the committed ncu capture
  verify        BASELINE config 3: verify_blob_kzg_proof_batch over 4096 blobs -- device-resident, pinned, pageable
  msm_sweep     BASELINE config 5: variable-base G1 MSM 2^12 .. 2^22, points/s and roofline fraction per size, next to
                the CPU restatement's g1_lincomb
  latency       single-call latency of every c-kzg entry point, GPU vs the CPU restatement
  cells         PeerDAS / EIP-7594 in the mainnet wire format: cells + FK20 cell proofs of 888 blobs (device-resident and
                through the host API), verify / recover latencies, checked against committed known answers
  cpu_baseline  the C restatement of the reference's CPU path (oracle/c) on a bounded sample of the same workload

--impl reference times that CPU restatement alone (the reference's own Rust code cannot be built here: no cargo,
un-vendored git dependencies); it never loads the product library.

--dump-outputs DIR writes what the last timed step returned to its caller -- commitments, proofs and status words --
as DIR/<name>.npy (see dump_outputs), so that two builds can be compared output for output on the same inputs.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BLOBS_PER_GPU = 1024
BLOB_BYTES = 4096 * 32
SETUP = os.path.join(ROOT, "tests", "golden", "trusted_setup.txt")
MAC32_PER_MSM = 2.80e8       # SURVEY §8d: fixed-base signed-digit bucket MSM-4096, c = 13: 933 888 Fp mul x 300 MAC32
MAC32_M, MAC32_S = 300.0, 234.0   # wide multiply-accumulates of one Fp product / square (csrc/mont.cuh)
IMAD_NOMINAL = 148 * 64 * 1.965e9  # SURVEY §8d sanity ceiling: one IMAD.WIDE per INT32 lane per clock
METRIC = "blobs/sec commit+proof"
UNIT = "blobs/s"
VERIFY_BLOBS = 4096
CELL_BLOBS = 888          # PeerDAS block: blobs per compute_cells_and_kzg_proofs batch (one pass; 888 x 128 = 113664 cell proofs)
# dram__bytes_read.sum + dram__bytes_write.sum of ONE 1024-blob launch of msm_gather_ba_kernel from the ncu --set full
# capture committed as profiles/r02_ncu_ba_1024blob_end_of_round_raw.csv
NCU_DRAM_BYTES_PER_BLOB = (35.41e9 + 9.30e9) / 1024
DUMP_LIMIT_BYTES = 64_000_000   # --dump-outputs: all ranks' files together


def workload_name(n, wb):
    return ("commit+proof (blob_to_kzg_commitment + compute_blob_kzg_proof) of %d synthetic 4096-element blobs per GPU, "
            "tests/golden/trusted_setup.txt (monomial, tau=1337), fixed-base window %d bits" % (n, wb))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().splitlines()[0]
                f = [x.strip() for x in out.split(",")]
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
                for nm, v in zip(names, f[2:]):
                    if v.lower().startswith("active"):
                        self.reasons.add(nm)
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------- CPU restatement
def cpu_reference_run(steps, warmup, sample_blobs=None):
    """Time the C restatement of the reference's CPU path with all host threads.  Uses oracle/ only."""
    from oracle import c_oracle

    oracle = c_oracle.COracle(open(SETUP).read())
    cores = oracle.max_threads()
    n = sample_blobs or max(16, 2 * cores)
    blobs = b"".join(oracle.synth_blob(k) for k in range(n))
    for _ in range(min(warmup, 1)):
        oracle.commit_and_prove_batch(blobs[: BLOB_BYTES * min(n, cores)], min(n, cores), cores)
    t0 = time.perf_counter()
    for _ in range(steps):
        rc, _, _ = oracle.commit_and_prove_batch(blobs, n, cores)
        assert rc == 0
    dt = (time.perf_counter() - t0) / steps
    return {"value": n / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "g1_msm_points_per_s": 2 * 4096 * n / dt,  # two MSM-4096 per blob dominate the CPU path as well
            "sample": "%d synthetic blobs per step (same generator as the GPU arm), one blob per thread, %d threads; "
                      "C restatement of the reference algorithm (per-call SRS re-hydration, Pippenger w=9, projective)" % (n, cores)}, dt


def cpu_latencies(oracle):
    """Single-call latency (ms) of the entry points the C restatement covers, one thread (the reference is
    single-threaded inside a call)."""
    blob = oracle.synth_blob(0)
    out = {}
    t = time.perf_counter(); rc, com = oracle.blob_to_kzg_commitment(blob); out["blob_to_kzg_commitment"] = (time.perf_counter() - t) * 1e3
    t = time.perf_counter(); oracle.compute_kzg_proof(blob, bytes(31) + b"\x05"); out["compute_kzg_proof"] = (time.perf_counter() - t) * 1e3
    t = time.perf_counter(); oracle.compute_blob_kzg_proof(blob, com); out["compute_blob_kzg_proof"] = (time.perf_counter() - t) * 1e3
    return out


def cpu_msm_points_per_s(oracle, lg):
    n = 1 << lg
    pts, sc = oracle.synth_msm_inputs(n, 1)
    t = time.perf_counter()
    rc, _ = oracle.g1_lincomb(pts, sc, n)
    dt = time.perf_counter() - t
    assert rc == 0
    return n / dt


# ---------------------------------------------------------------------------------------------- model helpers
def entries_per_point(wb, blob_fn, sample_blobs=2):
    """Average number of non-zero digits per SRS point (= table entries accumulated), counted on a small host-side
    sample with the kernel's own recoding rule (csrc/recode.cuh: GLV split, signed digits, unsigned top window)."""
    x2 = 0xD201000000010000 ** 2
    W = -(-128 // wb)
    nz = tot = 0
    for k in range(sample_blobs):
        blob = blob_fn(k)
        for i in range(0, len(blob), 32 * 16):  # every 16th word
            v = int.from_bytes(blob[i:i + 32], "big")
            for h in divmod(v, x2):
                carry = 0
                for j in range(W):
                    d = ((h >> (wb * j)) & ((1 << wb) - 1)) + carry
                    carry = 1 if (j < W - 1 and d > (1 << (wb - 1))) else 0
                    if carry:
                        d -= 1 << wb
                    nz += 1 if d != 0 else 0
            tot += 1
    return nz / tot


def var_msm_work_mac32(n):
    """SURVEY §8d work model for a variable-base MSM without precomputation."""
    return (min((255 // c + 1) * (10 * n + 14 * (1 << c)) for c in range(4, 24)) + 256 * 9) * 300.0


def dump_outputs(out_dir, first_blob, coms, proofs, status, ranks=1, suffix=""):
    """Write one step's outputs of a rank as DIR/<name><suffix>.npy, one row per blob: commitments.npy and proofs.npy
    (float32, n x 48, the byte values of the compressed G1 points), status.npy (float32, the C_KZG_RET of each blob)
    and blob_index.npy (float64, the synthetic blob number).  When the files of all ranks would exceed
    DUMP_LIMIT_BYTES, the same seeded sample of blobs is kept on every run."""
    import numpy as np

    n = len(status)
    rows = min(n, (DUMP_LIMIT_BYTES // ranks - 4096) // (4 * (48 + 48 + 1) + 8))   # 4096: room for the four .npy headers
    keep = np.arange(n) if rows == n else np.sort(np.random.default_rng(0).choice(n, rows, replace=False))
    arrays = {"commitments": np.frombuffer(coms, dtype=np.uint8).reshape(n, 48)[keep].astype(np.float32),
              "proofs": np.frombuffer(proofs, dtype=np.uint8).reshape(n, 48)[keep].astype(np.float32),
              "status": np.asarray(status)[keep].astype(np.float32),
              "blob_index": (first_blob + keep).astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--blobs", type=int, default=BLOBS_PER_GPU)
    ap.add_argument("--window-bits", type=int, default=16, help="fixed-base window c (16 -> 100 GiB table, the library default; shrinks automatically if HBM is short)")
    ap.add_argument("--no-extras", action="store_true", help="skip the verify / msm_sweep / latency blocks")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's commitments, proofs and status words to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs applies to --impl native")
    # Exactly ONE line on stdout (the JSON): native libraries (NCCL's version banner, CUDA warnings) write to fd 1
    # behind Python's back, so fd 1 is pointed at stderr for the whole run and the JSON goes to the saved descriptor.
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(json_fd, (json.dumps(obj) + "\n").encode())

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    n = args.blobs

    if args.impl == "reference":
        if rank != 0:
            return
        base, dt = cpu_reference_run(args.steps, args.warmup)
        line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": min(args.warmup, 1), "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u64 (6x64-bit Montgomery limbs)", "data": "synthetic",
                "config": {"workload": workload_name(n, args.window_bits) + "; CPU arm: bounded sample per step, see cpu_baseline.sample"},
                "cpu_baseline": base,
                "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        emit(line)
        return

    import torch
    import lambdaworks_kzg_b200 as lw

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    lw.set_option("window_bits", args.window_bits)
    settings = lw.load_trusted_setup_file(SETUP)
    wb = lw.window_bits(settings)
    stream = torch.cuda.current_stream().cuda_stream

    # ---- device-resident inputs: this rank's shard of the global synthetic batch
    blobs = torch.empty(n * BLOB_BYTES, dtype=torch.uint8, device=dev)
    lw.synth_blobs_device(blobs.data_ptr(), rank * n, n, stream)
    coms = torch.zeros(n * 48, dtype=torch.uint8, device=dev)
    proofs = torch.zeros(n * 48, dtype=torch.uint8, device=dev)
    status = torch.zeros(n, dtype=torch.int32, device=dev)

    def step():
        lw.commit_and_prove_batch_device(coms.data_ptr(), proofs.data_ptr(), blobs.data_ptr(), n, settings, stream, status.data_ptr())

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = lw.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    launches = lw.kernel_launches() - launches0
    ms = e0.elapsed_time(e1)
    assert int(status.abs().sum()) == 0
    ms_per_step = max_over_ranks(ms) / args.steps
    value = world * n / (ms_per_step * 1e-3)
    dev_coms, dev_proofs = bytes(coms.cpu().numpy().tobytes()), bytes(proofs.cpu().numpy().tobytes())
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, rank * n, dev_coms, dev_proofs, status.cpu().numpy(), world, "" if world == 1 else "_rank%d" % rank)

    # ---- end to end through the host-buffer C ABI call
    def e2e_run(h_blobs, h_coms, h_proofs):
        for _ in range(min(args.warmup, 2)):
            lw.commit_and_prove_batch(h_blobs.data_ptr(), n, settings, h_coms.data_ptr(), h_proofs.data_ptr())
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            st = lw.commit_and_prove_batch(h_blobs.data_ptr(), n, settings, h_coms.data_ptr(), h_proofs.data_ptr())
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / args.steps
        assert not any(st)
        assert bytes(h_coms.numpy().tobytes()) == dev_coms, "host-API and device-API commitments differ"
        assert bytes(h_proofs.numpy().tobytes()) == dev_proofs, "host-API and device-API proofs differ"
        return world * n / max_over_ranks(dt)

    host_blobs = blobs.cpu()                                    # pageable
    e2e_pageable = e2e_run(host_blobs, torch.zeros(n * 48, dtype=torch.uint8), torch.zeros(n * 48, dtype=torch.uint8))
    e2e_value = e2e_run(host_blobs.pin_memory(), torch.zeros(n * 48, dtype=torch.uint8).pin_memory(), torch.zeros(n * 48, dtype=torch.uint8).pin_memory())
    clocks = sampler.stop() if rank == 0 else None

    # ---- parity of what was just timed: a sample of THIS rank's outputs against the C restatement (checker only)
    from oracle import c_oracle

    oracle = c_oracle.COracle(open(SETUP).read())
    sample = sorted({0, n // 3, n // 2, n - 1})
    sb = b"".join(oracle.synth_blob(rank * n + k) for k in sample)
    rc, oc, op = oracle.commit_and_prove_batch(sb, len(sample), 0)
    mism = [k for i, k in enumerate(sample) if rc or dev_coms[48 * k:48 * k + 48] != oc[48 * i:48 * i + 48] or dev_proofs[48 * k:48 * k + 48] != op[48 * i:48 * i + 48]]
    bad_ranks = max_over_ranks(float(len(mism)))
    if bad_ranks:
        raise SystemExit("PARITY FAILURE: timed outputs differ from the oracle on rank %d, blobs %r" % (rank, mism))
    parity = {"checked_blobs_per_rank": len(sample), "ranks": world, "oracle": "oracle/c (C restatement), commitments and proofs byte-equal",
              "mismatches": 0}

    roofline = cpu_base = verify = msm_sweep = latency = None
    if rank == 0:
        # ---- roofline of the dominant kernel (measured alone, CUDA events on its own stream)
        k_ms = lw.bench_msm_kernel(blobs.data_ptr(), n, settings, 0, 5)
        peak = max(lw.imad_peak(1), lw.imad_peak(0))
        achieved = n * MAC32_PER_MSM / (k_ms * 1e-3)
        epp = entries_per_point(wb, oracle.synth_blob)  # table entries really accumulated per point
        alg_bytes = n * (BLOB_BYTES + 4096 * epp * 96)  # scalars streamed once + one 96 B table entry per non-zero digit
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        batch_affine = lw.get_option("msm_algo") == 1 and n >= lw.get_option("msm_ba_min_blobs")
        M, S = MAC32_M, MAC32_S
        if batch_affine:
            T, K = lw.get_option("msm_ba_threads"), lw.get_option("msm_ba_slots")
            rounds = -(-(4096 * epp / T) // K)
            floor_mac = n * 4096 * epp * (5 * M + S)            # this algorithm's own minimum: the affine additions alone
            executed = floor_mac + n * (T * (K - 1) * (8 * M + 2 * S)     # folding the K accumulators of a thread (XYZZ)
                                        + T * rounds * (20 * 120 + M)     # binary-GCD inversions: ~20 rounds x 120 wide MACs
                                        + (T - 1) * 14 * M)               # block tree
            kernel = "msm_gather_ba_kernel<BE, K=%d, threads=%d> (GLV halves, batched-affine accumulation, cp.async operand staging)" % (K, T)
        else:
            floor_mac = executed = n * 4096 * epp * (8 * M + 2 * S)
            kernel = "msm_gather_kernel<BE> (XYZZ accumulation)"
        traffic = n * NCU_DRAM_BYTES_PER_BLOB if batch_affine else None
        roofline = {"bound": "int32-imad", "kernel": kernel, "achieved": achieved / 1e12, "peak": peak / 1e12,
                    "unit": "TMAC32/s", "frac": achieved / peak,
                    "peak_source": "lwkzg_imad_peak(): memory-free IMAD.WIDE probe with distinct operand registers, run in this process "
                                   "(burst; best of carry-chain and carry-less variants; profiles/r01_pipe_probe.md). "
                                   "MEASURED_PEAKS.json carries no integer peak; the nominal figure is in peak_nominal",
                    "peak_nominal": IMAD_NOMINAL / 1e12,
                    "peak_note": "nominal = 148 SM x 64 INT32 lanes x 1.965 GHz (SURVEY 8d) assumes one IMAD.WIDE per lane per clock; a 32x32+64 MAC "
                                 "occupies the 16-lane fmaheavy pipe of an SM sub-partition for four cycles per warp whatever feeds it: 0.98 "
                                 "IMAD.WIDE per clock per SM even with an immediate multiplier and the multiplicand in the operand-reuse cache "
                                 "(round 1's 1.99 reading was ptxas hoisting the product out of the probe loop: profiles/r02_pipe_probe_imad_wide.md)",
                    "note": "achieved = SURVEY 8(d)'s ALGORITHMIC work (2.80e8 MAC32 per MSM-4096: bucket method, c = 13, XYZZ) / kernel time; "
                            "the kernel needs fewer multiplications than that model (full digit table, GLV, batched-affine additions), so frac may "
                            "exceed 1 -- frac_executed is the pipe-utilisation figure and frac_floor the distance to this algorithm's own minimum",
                    "alg_mac32_per_launch": n * MAC32_PER_MSM, "kernel_ms": k_ms,
                    "executed_mac32_per_launch": executed,
                    "frac_executed": executed / (k_ms * 1e-3) / peak,
                    "floor_mac32_per_launch": floor_mac,
                    "frac_floor": floor_mac / (k_ms * 1e-3) / peak,
                    "ncu_fmaheavy_pct": 74.6,
                    "ncu_source": "sm__pipe_fmaheavy_cycles_active of the 1024-blob launch (18.87 ms under ncu): profiles/r02_ncu_ba_1024blob_end_of_round_raw.csv",
                    "table_entries_per_point": epp,
                    "kernel_share_of_step": 2 * k_ms / ms_per_step,
                    # second half of BASELINE's metric: G1 MSM points/s (fixed-base MSM over the 4096-point SRS, this kernel)
                    "g1_msm_points_per_s": n * 4096 / (k_ms * 1e-3),
                    "traffic": traffic,
                    "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one 1024-blob launch, scaled to this launch's blob count "
                                      "(profiles/r02_ncu_ba_1024blob_end_of_round_raw.csv)",
                    "hbm": {"achieved": alg_bytes / (k_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                            "frac": alg_bytes / (k_ms * 1e-3) / 1e9 / hbm_peak, "alg_bytes_per_launch": alg_bytes,
                            "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s"}}

    if not args.no_extras:
        # ---- BASELINE config 3: batched verification of 4096 blobs per GPU
        verify = verify_block(lw, torch, dev, settings, rank, world, dist, barrier, max_over_ranks)
    if rank == 0 and not args.no_extras:
        # ---- BASELINE config 5: variable-base MSM sweep
        peak = roofline["peak"] * 1e12
        rows = []
        for lg in range(12, 23):
            m = 1 << lg
            ms_v, out = lw.bench_var_msm(m, settings, iters=5 if lg < 18 else 2, seed=1)
            rows.append({"log2_n": lg, "ms": ms_v, "points_per_s": m / (ms_v * 1e-3), "roofline_frac": var_msm_work_mac32(m) / (ms_v * 1e-3) / peak})
        cpu_pts = {}
        if world == 1:
            for lg in (12, 14):
                cpu_pts["2^%d" % lg] = cpu_msm_points_per_s(oracle, lg)
        # lwkzg_g1_lincomb itself (host buffers in, 48 bytes out): 4096 SRS points x random scalars
        g1v = settings.g1_values_bytes()
        be = lambda o: b"".join(g1v[o + 8 * q: o + 8 * q + 8][::-1] for q in range(6))  # noqa: E731  (6 x u64, most significant limb first)
        pts_be = b"".join(be(144 * i) + be(144 * i + 48) for i in range(4096))
        sc_be = bytes(blobs[:BLOB_BYTES].cpu().numpy().tobytes())
        lincomb_ms = {}
        for key, flag in (("any_curve_points", 0), ("points_in_g1", 1)):
            lw.set_option("lincomb_points_in_g1", flag)
            ref_out = lw.g1_lincomb(pts_be, sc_be, 4096)
            t0 = time.perf_counter()
            for _ in range(5):
                assert lw.g1_lincomb(pts_be, sc_be, 4096) == ref_out
            lincomb_ms[key] = (time.perf_counter() - t0) / 5 * 1e3
        lw.set_option("lincomb_points_in_g1", 0)
        assert ref_out == dev_coms[:48], "g1_lincomb(SRS, blob words) must be the blob's commitment"
        msm_sweep = {"sizes": rows, "cpu_g1_lincomb_points_per_s": cpu_pts,
                     "g1_lincomb_2^12_ms_per_call": lincomb_ms,
                     "g1_lincomb_note": "lwkzg_g1_lincomb from host buffers, H2D and D2H included; points_in_g1 = the caller vouches for subgroup "
                                        "membership (GLV split); the sweep itself runs on G1 points (table entries) with the split",
                     "cpu_note": "C restatement of g1_lincomb (unsigned Pippenger, homogeneous projective), one thread, as the reference runs it",
                     "work_model": "SURVEY 8d: min_c ceil(256/c) (10 N + 14 2^c) + 256*9 Fp products of 300 MAC32"}
        # ---- single-call latencies of the c-kzg entry points
        blob0 = bytes(blobs[:BLOB_BYTES].cpu().numpy().tobytes())
        c0, p0 = dev_coms[:48], dev_proofs[:48]
        z5 = bytes(31) + b"\x05"
        p5, y5 = lw.compute_kzg_proof(blob0, z5, settings)   # a true opening at z = 5: full-length scalars in the verification
        assert lw.verify_kzg_proof(c0, z5, y5, p5, settings) is True
        calls = [("blob_to_kzg_commitment", lambda: lw.blob_to_kzg_commitment(blob0, settings)),
                 ("compute_kzg_proof", lambda: lw.compute_kzg_proof(blob0, bytes(31) + b"\x05", settings)),
                 ("compute_blob_kzg_proof", lambda: lw.compute_blob_kzg_proof(blob0, c0, settings)),
                 ("verify_kzg_proof", lambda: lw.verify_kzg_proof(c0, z5, y5, p5, settings)),
                 ("verify_blob_kzg_proof", lambda: lw.verify_blob_kzg_proof(blob0, c0, p0, settings))]
        gpu_lat = {}
        for name, fn in calls:
            fn()
            t0 = time.perf_counter()
            for _ in range(5):
                fn()
            gpu_lat[name] = (time.perf_counter() - t0) / 5 * 1e3
        latency = {"unit": "ms per call", "gpu": gpu_lat, "cpu_restatement": cpu_latencies(oracle) if world == 1 else None,
                   "cpu_note": "oracle/c restates commit / proof only (no pairing), one thread: the reference is single-threaded inside a call"}
    cells = None
    if rank == 0 and not args.no_extras:
        cells = cells_block(lw, torch, dev, peak=roofline["peak"] * 1e12 if roofline else None)
    if rank == 0 and world == 1:
        cpu_base, _ = cpu_reference_run(1, 1)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u32 (12x32-bit Montgomery limbs, IMAD.WIDE)", "data": "synthetic",
                "config": {"workload": workload_name(n, wb), "blobs_per_gpu": n, "global_blobs": world * n, "parallelism": "blob-sharded x%d, no collective" % world,
                           "l2_policy": "inputs larger than L2: 128 MiB of blobs + random gathers from a %.1f GiB table per step" % (
                               sum(lw.table_geometry(wb)[1]) * 4096 * 96 / 2**30)},
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": n * BLOB_BYTES, "d2h_bytes_per_step": n * (48 + 48 + 4),
                        "api": "lwkzg_commit_and_prove_batch (host buffers, pinned)", "pageable_value": e2e_pageable,
                        "pageable_note": "same call from ordinary (pageable) host memory, what a c-kzg caller passes"},
                "gpu_launches": int(launches), "clocks": clocks, "parity": parity, "roofline": roofline, "verify": verify, "msm_sweep": msm_sweep,
                "latency": latency, "cells": cells, "cpu_baseline": cpu_base}
        emit(line)
    settings.free()
    if dist is not None:
        dist.destroy_process_group()


def cells_block(lw, torch, dev, n=CELL_BLOBS, peak=None):
    """PeerDAS / EIP-7594 (SURVEY 8 f4, include/lwkzg.h part 3) in the mainnet wire format (MODE_DENEB): cells + FK20 cell
    proofs of n device-resident blobs, the same through the host API, and the single-call latencies.  Checked against
    the committed known answers (tests/golden/cell_kats.json, made by the oracle without FK20) and by verifying a
    sample of the timed outputs with verify_cell_kzg_proof_batch."""
    import hashlib
    import random

    R = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
    lw.set_option("mode", 2)
    lw.set_option("window_bits", 8)    # the commitment table of these second settings stays small; the FK20 table is the one that matters
    t0 = time.perf_counter()
    s = lw.load_trusted_setup_file(SETUP)
    lw.set_option("mode", 0)
    try:
        kat = json.load(open(os.path.join(ROOT, "tests", "golden", "cell_kats.json")))[0]
        rng = random.Random(kat["seed"])
        blob = b"".join(rng.randrange(R).to_bytes(32, "big") for _ in range(4096))
        t1 = time.perf_counter()
        cs, ps = lw.compute_cells_and_kzg_proofs(blob, s)     # first call: builds the FK20 points and their digit table
        t_first = time.perf_counter() - t1
        assert hashlib.sha256(b"".join(cs)).hexdigest() == kat["cells_sha256"], "cells differ from the known answer"
        assert [ps[i].hex() for i in kat["proof_cells"]] == kat["proofs"], "cell proofs differ from the known answer"
        com = lw.blob_to_kzg_commitment(blob, s)
        stream = torch.cuda.current_stream().cuda_stream
        d_blobs = torch.empty(n * BLOB_BYTES, dtype=torch.uint8, device=dev)
        lw.synth_blobs_device(d_blobs.data_ptr(), 3 << 20, n, stream)
        d_cells = torch.zeros(n * 128 * 2048, dtype=torch.uint8, device=dev)
        d_proofs = torch.zeros(n * 128 * 48, dtype=torch.uint8, device=dev)
        d_st = torch.zeros(n, dtype=torch.int32, device=dev)

        def dev_ms(cells_ptr, proofs_ptr, reps=3):
            lw.compute_cells_and_kzg_proofs_batch_device(cells_ptr, proofs_ptr, d_blobs.data_ptr(), n, s, stream, d_st.data_ptr())
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                lw.compute_cells_and_kzg_proofs_batch_device(cells_ptr, proofs_ptr, d_blobs.data_ptr(), n, s, stream, d_st.data_ptr())
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / reps

        ms_both = dev_ms(d_cells.data_ptr(), d_proofs.data_ptr())
        ms_cells = dev_ms(d_cells.data_ptr(), 0)
        assert int(d_st.abs().sum()) == 0
        # host API, pinned buffers
        hb = d_blobs.cpu().pin_memory()
        hc = torch.zeros(n * 128 * 2048, dtype=torch.uint8).pin_memory()
        hp = torch.zeros(n * 128 * 48, dtype=torch.uint8).pin_memory()
        lib = lw.load_library()
        st = (ctypes.c_int * n)()
        host_call = lambda: lib.lwkzg_compute_cells_and_kzg_proofs_batch(hc.data_ptr(), hp.data_ptr(), hb.data_ptr(), n, s.ptr, st)  # noqa: E731
        assert host_call() == 0
        t2 = time.perf_counter()
        assert host_call() == 0
        ms_host = (time.perf_counter() - t2) * 1e3
        assert bytes(hp.numpy()) == bytes(d_proofs.cpu().numpy()) and bytes(hc.numpy()) == bytes(d_cells.cpu().numpy())
        # a sample of the timed outputs verifies in one batched check over n commitments; a swapped proof does not
        d_c = torch.zeros(n * 48, dtype=torch.uint8, device=dev)
        lw.blob_to_kzg_commitment_batch_device(d_c.data_ptr(), d_blobs.data_ptr(), n, s, stream, d_st.data_ptr())
        torch.cuda.synchronize()
        coms = bytes(d_c.cpu().numpy())
        cells_b, proofs_b = bytes(hc.numpy()), bytes(hp.numpy())
        rng = random.Random(1)
        pick = [(b, rng.randrange(128)) for b in range(n) for _ in range(2)]
        v_args = ([coms[48 * b: 48 * b + 48] for b, _ in pick], [i for _, i in pick],
                  [cells_b[(b * 128 + i) * 2048: (b * 128 + i + 1) * 2048] for b, i in pick],
                  [proofs_b[(b * 128 + i) * 48: (b * 128 + i + 1) * 48] for b, i in pick])
        assert lw.verify_cell_kzg_proof_batch(*v_args, s) is True
        swapped = list(v_args[3])
        swapped[0], swapped[1] = swapped[1], swapped[0]
        assert lw.verify_cell_kzg_proof_batch(v_args[0], v_args[1], v_args[2], swapped, s) is False

        def lat(fn, reps=3):
            fn()
            t = time.perf_counter()
            for _ in range(reps):
                fn()
            return (time.perf_counter() - t) / reps * 1e3

        keep = list(range(0, 128, 2))
        latency = {
            "compute_cells_and_kzg_proofs": lat(lambda: lw.compute_cells_and_kzg_proofs(blob, s)),
            "compute_cells_only": lat(lambda: lw.compute_cells_and_kzg_proofs(blob, s, want_proofs=False)),
            "recover_cells_and_kzg_proofs_64_of_128": lat(lambda: lw.recover_cells_and_kzg_proofs(keep, [cs[i] for i in keep], s)),
            "verify_cell_kzg_proof_batch_128_cells_1_blob": lat(lambda: lw.verify_cell_kzg_proof_batch([com] * 128, list(range(128)), cs, ps, s)),
            "verify_cell_kzg_proof_batch_%d_cells_%d_blobs" % (len(pick), n): lat(lambda: lw.verify_cell_kzg_proof_batch(*v_args, s), reps=2),
        }
        # executed integer work of a blob's 128 proofs (DESIGN 3.1): 8192 points x 2 GLV halves x W windows of batched-affine
        # additions (5 M + 1 S) + the fold of the accumulators, and 642 twiddle ladders of 129 Jacobian doublings (2 M + 5 S)
        # + ~52 mixed additions (7 M + 4 S) + the table of odd multiples
        cwb = lw.cell_window_bits(s)
        nwin = -(-128 // cwb)
        M, S = MAC32_M, MAC32_S
        mac_msm = 8192 * 2 * nwin * (1 - 2.0 ** -cwb) * (5 * M + S) + 2 * 128 * 63 * (8 * M + 2 * S)
        mac_fft = 642 * (129 * (2 * M + 5 * S) + 52 * (7 * M + 4 * S) + 3 * (2 * M + 5 * S) + 3 * (7 * M + 4 * S) + 40 * M)
        pk = peak or max(lw.imad_peak(1), lw.imad_peak(0))
        roof = {"bound": "int32-imad", "unit": "TMAC32/s", "peak": pk / 1e12,
                "achieved": n * (mac_msm + mac_fft) / (ms_both * 1e-3) / 1e12, "frac": n * (mac_msm + mac_fft) / (ms_both * 1e-3) / pk,
                "executed_mac32_per_blob": {"fk20_msm (msm_gather_ba_kernel, segmented)": mac_msm, "g1_fft (cell_g1_fft_stage_kernel)": mac_fft},
                "note": "whole pass (poly + toeplitz + 2 MSM launches + 14 FFT stage launches + finalize) against the measured integer-multiply "
                        "peak; per-kernel shares and ncu pipe utilisation: profiles/r02_cells_summary.md (fmaheavy 72 % MSM, 61-68 % FFT stages)"}
        return {"mode": "MODE_DENEB (mainnet wire format)", "blobs": n, "fk20_window_bits": lw.cell_window_bits(s), "roofline": roof,
                "setup_s": {"load_trusted_setup (Lagrange SRS + 8-bit commitment table)": t1 - t0, "first cell call (FK20 points + digit table)": t_first},
                "device_resident": {"cells_and_proofs_ms": ms_both, "cells_only_ms": ms_cells, "blobs_per_s": n / (ms_both * 1e-3),
                                    "cell_proofs_per_s": n * 128 / (ms_both * 1e-3)},
                "host_pinned": {"ms": ms_host, "blobs_per_s": n / (ms_host * 1e-3), "h2d_bytes": n * BLOB_BYTES, "d2h_bytes": n * 128 * (2048 + 48)},
                "latency_ms": latency,
                "parity": "known answers of tests/golden/cell_kats.json (oracle/py/cells.py, proofs computed without FK20); %d sampled cells of the timed "
                          "batch verify together and fail with two proofs swapped; host API bytes == device API bytes" % len(pick),
                "cpu_note": "no CPU figure: the reference implements no cell path (src/srs.rs:274 reads 2 of its 65 G2 points)"}
    finally:
        s.free()
        lw.set_option("window_bits", 16)


def verify_block(lw, torch, dev, settings, rank, world, dist, barrier, max_over_ranks):
    """verify_blob_kzg_proof_batch over VERIFY_BLOBS blobs per GPU (SURVEY §8d config 3): commitments / proofs come
    from our own commit+prove; the all-valid batch must verify and the batch with proof #n/2-1 replaced by another
    point must not.  At N > 1 every rank verifies its own batch (replicas: the numbers are per-GPU batches in
    flight at once) and the distributed check of the union of all batches is timed as well."""
    nv = VERIFY_BLOBS
    d_blobs = torch.empty(nv * BLOB_BYTES, dtype=torch.uint8, device=dev)
    lw.synth_blobs_device(d_blobs.data_ptr(), 1 << 20 | (rank * nv), nv, torch.cuda.current_stream().cuda_stream)
    d_c = torch.zeros(nv * 48, dtype=torch.uint8, device=dev)
    d_p = torch.zeros(nv * 48, dtype=torch.uint8, device=dev)
    d_st = torch.zeros(nv, dtype=torch.int32, device=dev)
    lw.commit_and_prove_batch_device(d_c.data_ptr(), d_p.data_ptr(), d_blobs.data_ptr(), nv, settings, torch.cuda.current_stream().cuda_stream, d_st.data_ptr())
    torch.cuda.synchronize()
    assert int(d_st.abs().sum()) == 0

    def timed(fn, reps=3):
        assert fn() is True
        barrier()
        best = 1e9
        for _ in range(reps):
            t0 = time.perf_counter()
            ok = fn()
            best = min(best, time.perf_counter() - t0)
            assert ok is True
        return max_over_ranks(best)

    out = {"blobs_per_gpu": nv, "unit": UNIT}
    t_dev = timed(lambda: lw.verify_blob_kzg_proof_batch_device(d_blobs.data_ptr(), d_c.data_ptr(), d_p.data_ptr(), nv, settings))
    bad = d_p.clone()
    bad[48 * (nv // 2 - 1): 48 * (nv // 2)] = d_c[:48]
    assert lw.verify_blob_kzg_proof_batch_device(d_blobs.data_ptr(), d_c.data_ptr(), bad.data_ptr(), nv, settings) is False
    out["device_resident"] = {"ms": t_dev * 1e3, "value": world * nv / t_dev}
    hb, hc, hp = d_blobs.cpu(), d_c.cpu(), d_p.cpu()
    t_page = timed(lambda: lw.verify_blob_kzg_proof_batch_ptr(hb.data_ptr(), hc.data_ptr(), hp.data_ptr(), nv, settings))
    out["pageable"] = {"ms": t_page * 1e3, "value": world * nv / t_page}
    pb, pc, pp = hb.pin_memory(), hc.pin_memory(), hp.pin_memory()
    t_pin = timed(lambda: lw.verify_blob_kzg_proof_batch_ptr(pb.data_ptr(), pc.data_ptr(), pp.data_ptr(), nv, settings))
    out["pinned"] = {"ms": t_pin * 1e3, "value": world * nv / t_pin, "h2d_bytes": nv * (BLOB_BYTES + 96)}
    out["corrupted_batch_rejected"] = True
    out["scaling_note"] = "device_resident / pinned / pageable: every rank verifies its OWN batch of %d blobs (independent batches, weak scaling)" % nv
    out["pairing_ms"] = lw.bench_pairing(settings, 5)   # partial-sum fold + 2-pairing check alone (CUDA events)
    if dist is not None and hasattr(lw, "verify_blob_kzg_proof_batch_distributed_device"):
        t_dist = timed(lambda: lw.verify_blob_kzg_proof_batch_distributed_device(d_blobs.data_ptr(), d_c.data_ptr(), d_p.data_ptr(), world * nv, settings,
                                                                                 inputs_on_device=True))
        out["distributed"] = {"ms": t_dist * 1e3, "value": world * nv / t_dist, "global_blobs": world * nv,
                              "note": "ONE batch of world x %d device-resident blobs sharded over the ranks; two all-gathers (160 B per blob, 288 B per "
                                      "rank) over NCCL on device tensors.  Bounded by the batch challenge r: one sequential SHA-256 over all "
                                      "world x %d tuples (~2.5 us per blob on one GPU lane), which no number of GPUs shortens -- the per-GPU "
                                      "batches above are what scales" % (nv, nv)}
    return out


if __name__ == "__main__":
    main()
