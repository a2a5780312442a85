#!/usr/bin/env python3
"""One process per GPU over NCCL (SURVEY §8e):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P tools/multi_gpu_check.py

Runs twice: with NB synthetic blobs, and with NB + 3 (2051 by default: uneven shards for 2, 4 and 8 ranks).
* every rank commits to and proves its contiguous shard of the blobs (no communication); rank 0 recomputes the
  whole batch alone and the shard outputs must be byte-equal to it;
* the batch is verified three ways -- monolithic on rank 0, distributed with host exchanges (gloo-style bytes path) and
  distributed with every exchanged byte in device memory -- and all must agree, also after corrupting one proof;
* both distributed drivers must reject a forged proof pair at the same local index of ranks 0 and 1 (it passes if the
  two items get the same weight, i.e. if a rank's offset in the batch were ignored: tests/_forge.py).
Prints MULTI_GPU_CHECK_OK on success."""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch, torch.distributed as dist
import lambdaworks_kzg_b200 as lw
from oracle.py import kzg
from tests import _forge

rank, local, world = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
NB = int(os.environ.get("NB", "2048"))
lw.set_option("window_bits", int(os.environ.get("WB", "13")))
setup_path = os.path.join(ROOT, "tests", "golden", "trusted_setup.txt")
s = lw.load_trusted_setup_file(setup_path)
ref = kzg.RefMode(kzg.parse_setup_text(open(setup_path).read()))
dev = torch.device("cuda", local)
B = 131072


def check(n_total):
    first, cnt = lw.shard_range(n_total, world, rank)
    d_blobs = torch.empty(cnt * B, dtype=torch.uint8, device=dev)
    lw.synth_blobs_device(d_blobs.data_ptr(), first, cnt, 0)
    torch.cuda.synchronize()
    blobs = bytes(d_blobs.cpu().numpy().tobytes())
    coms, proofs, st = lw.commit_and_prove_batch(blobs, cnt, s)
    assert not any(st)
    outs = [None] * world
    dist.all_gather_object(outs, (coms, proofs))
    all_c = [c for o in outs for c in o[0]]
    all_p = [p for o in outs for p in o[1]]
    if rank == 0:
        full = torch.empty(n_total * B, dtype=torch.uint8, device=dev)
        lw.synth_blobs_device(full.data_ptr(), 0, n_total, 0)
        torch.cuda.synchronize()
        full_b = bytes(full.cpu().numpy().tobytes())
        c1, p1, st1 = lw.commit_and_prove_batch(full_b, n_total, s)
        assert not any(st1)
        assert c1 == all_c and p1 == all_p, "shard outputs differ from the single-GPU outputs"
        mono = lw.verify_blob_kzg_proof_batch([full_b[i * B:(i + 1) * B] for i in range(n_total)], all_c, all_p, s)
        assert mono is True
        del full
    dist.barrier()
    cb, pb = b"".join(coms), b"".join(proofs)
    ok_host = lw.verify_blob_kzg_proof_batch_distributed(blobs, cb, pb, n_total, s)
    d_c = torch.frombuffer(bytearray(cb), dtype=torch.uint8).to(dev)
    d_p = torch.frombuffer(bytearray(pb), dtype=torch.uint8).to(dev)
    torch.cuda.synchronize(); dist.barrier()
    times = []
    for rep in range(3):
        t0 = time.perf_counter()
        ok_dev = lw.verify_blob_kzg_proof_batch_distributed_device(d_blobs.data_ptr(), d_c.data_ptr(), d_p.data_ptr(), n_total, s, inputs_on_device=True)
        torch.cuda.synchronize(); dist.barrier()
        times.append((time.perf_counter() - t0) * 1e3)

    def both(proof_list):
        d = torch.frombuffer(bytearray(b"".join(proof_list)), dtype=torch.uint8).to(dev)
        torch.cuda.synchronize()
        ok_d = lw.verify_blob_kzg_proof_batch_distributed_device(d_blobs.data_ptr(), d_c.data_ptr(), d.data_ptr(), n_total, s, inputs_on_device=True)
        ok_h = lw.verify_blob_kzg_proof_batch_distributed(blobs, cb, b"".join(proof_list), n_total, s)
        return ok_d, ok_h

    bad = list(proofs)
    if rank == world - 1:
        bad[-1] = coms[0]
    ok_bad = both(bad)
    ok_forged = (False, False)
    if world >= 2:
        # the forged pair: local index 5 of ranks 0 and 1 (every rank derives the same pair)
        i, j = 5, lw.shard_range(n_total, world, 1)[0] + 5
        pi, pj = _forge.forge_pair(all_p[i], all_p[j], _forge.blob_factor(ref, lw.synth_blob_host(i), all_c[i]),
                                   _forge.blob_factor(ref, lw.synth_blob_host(j), all_c[j]))
        forged = list(proofs)
        for k, p in ((i, pi), (j, pj)):
            if first <= k < first + cnt:
                forged[k - first] = p
        ok_forged = both(forged)
    assert ok_host is True and ok_dev is True and ok_bad == (False, False) and ok_forged == (False, False), (ok_host, ok_dev, ok_bad, ok_forged)
    if rank == 0:
        print("world=%d n=%d: shard outputs == single GPU, distributed verify (host / device exchanges) == monolithic%s; "
              "device-resident distributed verify %.1f ms (best of 3)" % (world, n_total, ", forged pair rejected" if world >= 2 else "", min(times)),
              flush=True)


for n in (NB, NB + 3):
    check(n)
if rank == 0:
    print("MULTI_GPU_CHECK_OK", flush=True)
dist.destroy_process_group()
