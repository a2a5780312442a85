"""bench.py --dump-outputs: the files it writes (format, size limit, seeded sample) and, on the GPU, that they hold what
the timed step computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SETUP = os.path.join(ROOT, "tests", "golden", "trusted_setup.txt")


def _fake_step(n):
    rng = np.random.default_rng(5)
    return rng.integers(0, 256, n * 48, dtype=np.uint8).tobytes(), rng.integers(0, 256, n * 48, dtype=np.uint8).tobytes(), \
        rng.integers(0, 2, n, dtype=np.int32)


def _load(d, suffix=""):
    return {k: np.load(os.path.join(d, k + suffix + ".npy")) for k in ("commitments", "proofs", "status", "blob_index")}


def test_dump_outputs_writes_every_blob(tmp_path):
    coms, proofs, status = _fake_step(10)
    bench.dump_outputs(str(tmp_path), 100, coms, proofs, status)
    a = _load(tmp_path)
    assert a["commitments"].dtype == np.float32 and a["commitments"].shape == (10, 48)
    assert a["proofs"].dtype == np.float32 and a["proofs"].shape == (10, 48)
    assert a["status"].dtype == np.float32 and a["status"].tolist() == status.tolist()
    assert a["blob_index"].dtype == np.float64 and a["blob_index"].tolist() == list(range(100, 110))
    assert a["commitments"].astype(np.uint8).tobytes() == coms and a["proofs"].astype(np.uint8).tobytes() == proofs


def test_dump_outputs_samples_within_the_limit(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 1 << 20)
    n, ranks = 5000, 2
    coms, proofs, status = _fake_step(n)
    for d in ("a", "b"):
        for r in range(ranks):
            bench.dump_outputs(str(tmp_path / d), r * n, coms, proofs, status, ranks, "_rank%d" % r)
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 1 << 20
    a0, b0 = _load(tmp_path / "a", "_rank0"), _load(tmp_path / "b", "_rank0")
    for k in a0:
        assert np.array_equal(a0[k], b0[k]), "the sample must be the same on every run"
    idx = a0["blob_index"].astype(np.int64)
    assert 0 < len(idx) < n and np.all(np.diff(idx) > 0)
    rows = np.frombuffer(coms, dtype=np.uint8).reshape(n, 48)[idx]
    assert np.array_equal(a0["commitments"], rows.astype(np.float32))
    assert np.array_equal(_load(tmp_path / "a", "_rank1")["blob_index"], a0["blob_index"] + n)


@pytest.mark.gpu
def test_bench_dump_outputs_match_the_oracle(tmp_path):
    from oracle import c_oracle

    n, steps = 6, 2
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1", "--blobs", str(n),
           "--window-bits", "8", "--no-extras", "--dump-outputs", str(tmp_path)]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-4000:]
    lines = p.stdout.splitlines()
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == steps
    a = _load(tmp_path)
    assert a["status"].tolist() == [0.0] * n and a["blob_index"].tolist() == list(range(n))
    oracle = c_oracle.COracle(open(SETUP).read())
    rc, oc, op = oracle.commit_and_prove_batch(b"".join(oracle.synth_blob(k) for k in range(n)), n, 0)
    assert rc == 0
    assert a["commitments"].astype(np.uint8).tobytes() == oc
    assert a["proofs"].astype(np.uint8).tobytes() == op
