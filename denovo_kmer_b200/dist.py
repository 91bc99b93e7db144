"""Multi-GPU plumbing: one process per GPU, read batches sharded across ranks, the
spanning-k-mer table replicated, and ONE sum-allreduce of the per-entry count vector
(north_star; SURVEY.md §8e).  No other collective exists on the path, and it is made by
libdkb.so itself (dkb_comm_init / dkb_counts_allreduce / dkb_reduce_push: ncclAllReduce on
the library's streams).  This module only shards the work and hands the NCCL id round.
"""
import os

import numpy as np


def env_rank_world():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(
        os.environ.get("LOCAL_RANK", 0))


def shard_range(n_items: int, rank: int, world: int):
    """Contiguous, balanced slice [lo, hi) of n_items read batches (or reads) for rank."""
    base, rem = divmod(n_items, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class _DevArray:
    """Expose a raw device pointer through __cuda_array_interface__ (int32 view)."""

    def __init__(self, ptr: int, n: int):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<i4", "data": (ptr, False),
                                         "version": 2}


def counts_tensor(kc):
    """torch int32 view (no copy) of the context's [n_samples][n_entries] device counters (tests and
    checks; the product's own sum over ranks never leaves the library)."""
    import torch
    ptr, n = kc.entry_counts_device()
    if n == 0:
        return torch.zeros(0, dtype=torch.int32, device=f"cuda:{kc.device}")
    return torch.as_tensor(_DevArray(ptr, n), device=f"cuda:{kc.device}")


def bootstrap_comm(kc, rank: int, world: int, group=None):
    """Give the context its NCCL communicator (inside libdkb.so).  The 128-byte id is made by
    rank 0 and handed round with one torch.distributed broadcast on whatever process group
    the launcher set up (gloo or nccl) - bootstrap only; the counters never go through torch."""
    if world == 1:
        return
    import torch.distributed as tdist
    from . import api
    box = [api.comm_unique_id() if rank == 0 else None]
    tdist.broadcast_object_list(box, src=0, group=group)
    kc.comm_init(box[0], rank, world)


def allreduce_counts_numpy(counts: np.ndarray, group=None) -> np.ndarray:
    """Host-side sum over ranks (gloo tests of the sharding logic): uint32/uint64 array ->
    summed copy.  The GPU path does not use this: its sum is ncclAllReduce inside the library."""
    import torch
    import torch.distributed as tdist
    t = torch.from_numpy(counts.astype(np.int64))
    if tdist.is_available() and tdist.is_initialized() and tdist.get_world_size(group) > 1:
        tdist.all_reduce(t, op=tdist.ReduceOp.SUM, group=group)
    return t.numpy().astype(counts.dtype)


class CountPipeline:
    """Overlap the sum over ranks of one batch's counters with the scan of the next batch -
    a thin caller of dkb_reduce_push / dkb_reduce_flush (the double-buffered snapshot, the
    side stream and the ncclAllReduce all live in libdkb.so).

    push() - call it when a batch's scans have been submitted - snapshots the counters and
    starts their sum; the PREVIOUS batch is finalised (kernel 3) behind this batch's scans.
    flush() finalises the last batch.  Without a communicator (one GPU) the results equal
    plain finalise()."""

    def __init__(self, kc, thresholds):
        self.kc, self.thr = kc, thresholds

    def push(self):
        self.kc.reduce_push(self.thr)

    def flush(self):
        self.kc.reduce_flush(self.thr)
