"""Multi-GPU plumbing: env instances are sharded across ranks (no data-path collective); the only exchanges are
the PPO gradient all-reduce, the (sum, sum of squares) of the return statistics, and the HAPPO agent order (plus, at a
training-state checkpoint, one broadcast and two all-reduces of a failure count).
Works over NCCL (one rank per GPU) and over gloo on CPU tensors (the world_size-2 tests)."""
from __future__ import annotations

import os

import numpy as np
import torch
import torch.distributed as dist


def active():
    return dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1


def rank():
    return dist.get_rank() if active() else 0


def world_size():
    return dist.get_world_size() if active() else 1


def all_reduce_sum_(t):
    """In-place sum over ranks (NVLink / NVSwitch through NCCL on device tensors)."""
    if active():
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t


def broadcast_order(order, device):
    """Every rank must apply the same HAPPO agent cycle (d2d_ppo.py:421-422): rank 0's shuffle wins."""
    t = torch.as_tensor(np.asarray(order, dtype=np.int32)).to(device)
    if active():
        dist.broadcast(t, src=0)
    return t


def broadcast_token(device):
    """A random 48-bit integer drawn by rank 0 and shared by every rank (names the files of one checkpoint)."""
    t = torch.tensor([int.from_bytes(os.urandom(6), "little")], dtype=torch.int64, device=device)
    if active():
        dist.broadcast(t, src=0)
    return int(t.item())


def shard(n_total, r=None, w=None):
    """Contiguous block of the global env index space owned by rank r: (offset, count)."""
    r = rank() if r is None else r
    w = world_size() if w is None else w
    base, rem = divmod(int(n_total), w)
    count = base + (1 if r < rem else 0)
    offset = r * base + min(r, rem)
    return offset, count


def is_last_shard():
    return rank() == world_size() - 1


def merge_moments(stats, n_local, ddof):
    """Global mean / std of columns from per-rank [cols, 2] (sum, sum of squares) and the local row count."""
    s = stats.clone()
    n = torch.tensor([float(n_local)], dtype=torch.float64, device=s.device)
    all_reduce_sum_(s)
    all_reduce_sum_(n)
    n = n.item()
    mean = s[:, 0] / n
    var = (s[:, 1] - n * mean * mean) / (n - ddof)
    return mean, var.clamp(min=0).sqrt()
