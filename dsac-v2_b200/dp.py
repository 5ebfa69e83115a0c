"""Data-parallel seam of the update path (SURVEY.md §8e): replicate the six networks,
shard the minibatch across ranks, exchange

  1. the two per-critic sums of std (inputs of the mean_std EMA that every sample's
     TD bound and gradient weight depend on, reference dsac_v2.py:233-241) — 2 floats, SUM;
  2. the flat gradient buffer [q1 | q2 | policy | log_alpha] — one all-reduce, SUM
     (each rank already scales its loss terms by 1/global_batch);
  3. the logged accumulators (16 sums, 2 minima).

Two transports.  `connect_peers` + `engine.dp_step`: the exchanges run inside the step's own
kernels over NVLink peer memory (CUDA IPC), the whole data-parallel step is one graph launch
per rank.  `data_parallel_gradients`: the same seam through `torch.distributed` (NCCL on
GPUs; gloo in the CPU tests) — the fallback, and the path of the split gradient API.  `engine` is anything with grad_phase1 / grad_phase2 / state / grads — the CUDA
`Engine`, the head-wise `CnnEngine` (which has no peer-memory exchange: this is its only data-parallel path), or a
CPU stand-in in tests/test_dp_gloo.py.
"""
from __future__ import annotations

from . import _lib


def world(dist_module=None):
    """(dist, world_size) if a multi-rank process group is live, else (None, 1)."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        return dist, dist.get_world_size()
    return None, 1


def shard_rows(n_rows: int, rank: int, world_size: int):
    """Contiguous [lo, hi) slice of a global minibatch owned by `rank` (sizes differ by at most 1)."""
    base, rem = divmod(n_rows, world_size)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def data_parallel_gradients(engine, data, noise, dist, local_rows: int, global_rows: int) -> int:
    """Forward, exchange std sums, losses + backward with means over `global_rows`, exchange gradients."""
    engine.grad_phase1(data, noise)
    dist.all_reduce(engine.state[_lib.STATE_STDSUM:_lib.STATE_STDSUM + 2])
    engine.grad_phase2(global_rows)
    dist.all_reduce(engine.grads)
    dist.all_reduce(engine.state[_lib.STATE_ACC:_lib.STATE_ACC + 16])
    dist.all_reduce(engine.state[_lib.STATE_ACC + 16:_lib.STATE_ACC + 18], op=dist.ReduceOp.MIN)
    return global_rows


def connect_peers(engine, dist) -> bool:
    """Map the ranks' exchange buffers into each other (CUDA IPC) so that `engine.dp_step` can run the exchanges inside
    the step's own kernels (include/dsact.h, csrc/dp_peer.cuh).  Collective: every rank must call it.  Returns False —
    on every rank alike — if any rank cannot export or map a buffer (no peer access, IPC disabled in the container,
    more than DSACT_DP_MAX_RANKS ranks); the caller then stays on the NCCL path above."""
    world_size, rank = dist.get_world_size(), dist.get_rank()
    handle, err = None, None
    if world_size > _lib.DP_MAX_RANKS:
        err = f"world size {world_size} > {_lib.DP_MAX_RANKS}"
    else:
        try:
            handle = engine.dp_export()
        except _lib.DsactError as e:
            err = str(e)
    gathered = [None] * world_size
    dist.all_gather_object(gathered, (handle, err))
    ok = all(e is None for _, e in gathered)
    if ok:
        try:
            engine.dp_connect(rank, [h for h, _ in gathered])
        except _lib.DsactError as e:
            ok, err = False, str(e)
    flags = [None] * world_size
    dist.all_gather_object(flags, ok)     # also the barrier that dsact_dp_connect asks for
    if not all(flags):
        engine.dp_world = 0
        return False
    return True


def global_rows(dist, local_rows: int, device) -> int:
    """Sum of the ranks' shard sizes (ranks may hold ragged shards)."""
    import torch
    t = torch.tensor([local_rows], dtype=torch.int64, device=device)
    dist.all_reduce(t)
    return int(t.item())
