"""Multi-GPU partitioning: one process per GPU, filters sharded across ranks.

The filters of a batch are independent (no reference function couples two `filter` structs), so
the step needs NO data-path collective; the only exchanges are the gathers of per-filter statistics
(inlier counts, hypotheses run, status bits) and of the evaluation records (errors and NEES against the ground truth)
after a frame or a run — a few int32 / float64 per filter.
``torch.distributed`` is the plumbing: backend "nccl" on the GPU box (device tensors over
NVLink/NVSwitch), "gloo" in the CPU tests.
"""
from __future__ import annotations

import numpy as np

from ._lib import EVAL_FIELDS, STATS_FIELDS


def partition(n_filters, world_size, rank):
    """Contiguous block partition of filter indices: returns (b0, nb) of `rank`; the first
    ``n_filters % world_size`` ranks own one filter more."""
    if world_size <= 0 or not (0 <= rank < world_size):
        raise ValueError("bad world_size / rank")
    base, rem = divmod(n_filters, world_size)
    nb = base + (1 if rank < rem else 0)
    b0 = rank * base + min(rank, rem)
    return b0, nb


def _gather_rows(local, torch_dtype, n_filters_total, device, group):
    """All-gather of per-filter rows local [nb, F] over the ranks, in rank (= global filter) order."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return local
    world = dist.get_world_size(group)
    dev = device if device is not None else ("cuda" if dist.get_backend(group) == "nccl" else "cpu")
    counts = torch.zeros(world, dtype=torch.int64, device=dev)
    counts[dist.get_rank(group)] = local.shape[0]
    dist.all_reduce(counts, group=group)
    nmax = int(counts.max().item())
    buf = torch.zeros((nmax, local.shape[1]), dtype=torch_dtype, device=dev)
    buf[:local.shape[0]] = torch.from_numpy(local).to(dev)
    out = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(out, buf, group=group)
    parts = [o[:int(c)].cpu().numpy() for o, c in zip(out, counts.tolist())]
    rows = np.concatenate(parts, axis=0)
    if n_filters_total is not None and rows.shape[0] != n_filters_total:
        raise RuntimeError("gathered %d filters, expected %d" % (rows.shape[0], n_filters_total))
    return rows


def gather_stats(stats, n_filters_total=None, device=None, group=None):
    """All-gathers the per-filter statistics dict of FilterBank.download_stats() over the ranks.
    Returns {field: int32 array [n_filters_total]} in global filter order on every rank."""
    import torch
    local = np.stack([np.asarray(stats[k], dtype=np.int32) for k in STATS_FIELDS], axis=1)  # [nb, F]
    allst = _gather_rows(local, torch.int32, n_filters_total, device, group)
    return {k: allst[:, i].copy() for i, k in enumerate(STATS_FIELDS)}


def gather_eval(rec, n_filters_total=None, device=None, group=None):
    """All-gathers the evaluation records of FilterBank.download_eval() (a frame's records or the running totals)
    over the ranks.  Returns {field: float64 array [n_filters_total]} in global filter order on every rank; the int32
    fields (n_map, n_skip, frames, status) are exact in float64."""
    import torch
    local = np.stack([np.asarray(rec[k], dtype=np.float64) for k in EVAL_FIELDS], axis=1)  # [nb, F]
    allrec = _gather_rows(local, torch.float64, n_filters_total, device, group)
    return {k: allrec[:, i].copy() for i, k in enumerate(EVAL_FIELDS)}


def max_over_ranks(value, device=None, group=None):
    """MAX-reduce of a python float over the ranks (timings are reported as the slowest rank)."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return float(value)
    dev = device if device is not None else ("cuda" if dist.get_backend(group) == "nccl" else "cpu")
    t = torch.tensor([float(value)], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return float(t.item())
