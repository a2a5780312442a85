"""Blob sharding across GPUs (one process per GPU) and the only exchange step the
hot path has: batched verification (SURVEY.md §8e).

commit / proof batches shard as contiguous ranges with NO communication.
verify_blob_kzg_proof_batch needs two tiny exchanges because the random
challenge r hashes every (C_i, z_i, y_i, pi_i) tuple (/root/reference/src/
utils.rs:166-206):

  phase 1 (local)   per blob: decode, z_i = challenge, y_i = p_i(z_i) -> 160-byte tuple
  exchange A        all_gather of the tuples (160 B per blob)
  phase 2 (local)   r, then partial sums over the rank's own index range (3 points, 288 B)
  exchange B        all_gather of the partial sums
  phase 3           add the partial sums, one 2-pairing check (identical on every rank)

Group addition is exact, so the boolean is independent of the number of ranks.
The collectives go through torch.distributed (NCCL over NVLink on the GPU box,
gloo in the CPU tests).  On the GPU box the exchanged data never leaves device
memory: verify_blob_kzg_proof_batch_distributed_device has phase 1 write its
tuples straight into the all-gather's input tensor (lwkzg_verify_batch_phase*_device).

What bounds one batch spread over many GPUs is not the exchange but r itself: a
single sequential SHA-256 over all n x 160 tuple bytes (~1 us per 64-byte block on
one GPU lane).  Independent batches per GPU scale linearly; one batch does not.
"""
from __future__ import annotations

from typing import Callable, Optional, Tuple

from . import api


def shard_range(n_total: int, world_size: int, rank: int) -> Tuple[int, int]:
    """Contiguous shard [first, first+count) of n_total items for `rank`."""
    base, rem = divmod(n_total, world_size)
    count = base + (1 if rank < rem else 0)
    first = rank * base + min(rank, rem)
    return first, count


class _CabiPhases:
    """Default compute backend: the C ABI of liblwkzg_b200.so."""

    def __init__(self, settings):
        self.s = settings

    def phase1(self, blobs, commitments, proofs, n_local):
        return api.verify_batch_phase1(blobs, commitments, proofs, n_local, self.s)

    def phase2(self, all_tuples, n_total, first, n_local):
        return api.verify_batch_phase2(all_tuples, n_total, first, n_local, self.s)

    def phase3(self, partials, n_ranks):
        return api.verify_batch_phase3(partials, n_ranks, self.s)

    def single(self, blob, commitment, proof):
        return api.verify_blob_kzg_proof(blob, commitment, proof, self.s)


def _all_gather_bytes(dist, payload: bytes, device) -> list:
    """all_gather of variable-length byte strings (sizes first, then padded data)."""
    import torch

    world = dist.get_world_size()
    size = torch.tensor([len(payload)], dtype=torch.int64, device=device)
    sizes = [torch.zeros(1, dtype=torch.int64, device=device) for _ in range(world)]
    dist.all_gather(sizes, size)
    sizes = [int(t.item()) for t in sizes]
    mx = max(max(sizes), 1)
    buf = torch.zeros(mx, dtype=torch.uint8, device=device)
    if payload:
        buf[: len(payload)] = torch.frombuffer(bytearray(payload), dtype=torch.uint8).to(device)
    outs = [torch.zeros(mx, dtype=torch.uint8, device=device) for _ in range(world)]
    dist.all_gather(outs, buf)
    return [bytes(o[:sz].cpu().numpy().tobytes()) for o, sz in zip(outs, sizes)]


def verify_blob_kzg_proof_batch_distributed(blobs_local: bytes, commitments_local: bytes, proofs_local: bytes, n_total: int,
                                            settings=None, *, dist=None, device=None, phases=None) -> bool:
    """verify_blob_kzg_proof_batch (lib.rs:525-614) with the batch sharded over
    the ranks of `dist` (default: torch.distributed's default group); this rank
    passes its own contiguous shard (see shard_range).  Returns the same
    boolean on every rank; raises KzgError on every rank if any rank saw an
    invalid item."""
    import torch

    if dist is None:
        import torch.distributed as dist  # type: ignore
    world, rank = dist.get_world_size(), dist.get_rank()
    if device is None:
        device = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
    ph = phases if phases is not None else _CabiPhases(settings)
    first, n_local = shard_range(n_total, world, rank)
    assert len(blobs_local) == n_local * api.BYTES_PER_BLOB

    if n_total == 0:
        # lib.rs:538-543: the reference rejects an empty batch; c-kzg (MODE_CKZG_LE) accepts it
        return api.get_option("mode") != 0 if phases is None else False
    err = 0
    tuples = b""
    result = False
    if n_total == 1:
        # lib.rs:544: single-blob path, run by the rank that owns the item
        if n_local == 1:
            try:
                result = ph.single(blobs_local, commitments_local, proofs_local)
            except api.KzgError as e:
                err = e.code
        flag = torch.tensor([err, int(result)], dtype=torch.int64, device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MAX)
        if int(flag[0]):
            raise api.KzgError(int(flag[0]), "verify_blob_kzg_proof_batch_distributed", "invalid item on some rank")
        return bool(int(flag[1]))

    try:
        tuples = ph.phase1(blobs_local, commitments_local, proofs_local, n_local) if n_local else b""
    except api.KzgError as e:
        err = e.code
    flag = torch.tensor([err], dtype=torch.int64, device=device)
    dist.all_reduce(flag, op=dist.ReduceOp.MAX)
    if int(flag[0]):
        raise api.KzgError(int(flag[0]), "verify_blob_kzg_proof_batch_distributed", "invalid item on some rank")
    all_tuples = b"".join(_all_gather_bytes(dist, tuples, device))  # exchange A
    assert len(all_tuples) == 160 * n_total
    partial = ph.phase2(all_tuples, n_total, first, n_local) if n_local else bytes(288)
    partials = b"".join(_all_gather_bytes(dist, partial, device))  # exchange B
    return ph.phase3(partials, world)


def verify_blob_kzg_proof_batch_distributed_device(blobs_ptr: int, commitments_ptr: int, proofs_ptr: int, n_total: int, settings, *,
                                                   inputs_on_device: bool, dist=None) -> bool:
    """The same protocol over NCCL with every exchanged byte in device memory.  blobs / commitments / proofs are raw
    addresses of THIS rank's contiguous shard (shard_range), in host memory or -- inputs_on_device -- on this rank's GPU.
    Needs n_total >= 2 (the single-blob path has nothing to shard)."""
    import torch

    if dist is None:
        import torch.distributed as dist  # type: ignore
    assert n_total >= 2
    world, rank = dist.get_world_size(), dist.get_rank()
    device = torch.device("cuda", torch.cuda.current_device())
    first, n_local = shard_range(n_total, world, rank)
    n_max = shard_range(n_total, world, 0)[1]   # rank 0 holds a largest shard
    # The library works on streams of its own that do not order after torch's: every tensor it reads or writes is
    # finished on torch's stream (allocated, zero-filled, gathered, concatenated) before the call.  A zero-fill that
    # landed after phase 2 would erase this rank's partial sums and drop its items from the pairing check.
    sync = torch.cuda.current_stream().synchronize
    mine = torch.zeros(n_max * 160, dtype=torch.uint8, device=device)
    err = 0
    try:
        if n_local:
            sync()
            api.verify_batch_phase1_device(mine.data_ptr(), blobs_ptr, commitments_ptr, proofs_ptr, n_local, settings, inputs_on_device)
    except api.KzgError as e:
        err = e.code
    flag = torch.tensor([err], dtype=torch.int64, device=device)
    dist.all_reduce(flag, op=dist.ReduceOp.MAX)
    if int(flag[0]):
        raise api.KzgError(int(flag[0]), "verify_blob_kzg_proof_batch_distributed_device", "invalid item on some rank")
    gathered = torch.empty(world * n_max * 160, dtype=torch.uint8, device=device)
    dist.all_gather_into_tensor(gathered, mine)                       # exchange A
    if n_total == world * n_max:
        all_tuples = gathered
    else:                                                             # uneven shards: drop the padding
        parts = [gathered[r * n_max * 160: r * n_max * 160 + shard_range(n_total, world, r)[1] * 160] for r in range(world)]
        all_tuples = torch.cat(parts)
    partial = torch.zeros(288, dtype=torch.uint8, device=device)
    if n_local:
        sync()
        api.verify_batch_phase2_device(partial.data_ptr(), all_tuples.data_ptr(), n_total, first, n_local, settings)
    partials = torch.empty(world * 288, dtype=torch.uint8, device=device)
    dist.all_gather_into_tensor(partials, partial)                    # exchange B
    sync()
    return api.verify_batch_phase3_device(partials.data_ptr(), world, settings)
