"""Multi-GPU partitioning of independent evaluations (hyper-parameter draws, per-group GPs).

The reference parallelises exactly this axis with OS processes: mclapply(s_list, ..., mc.cores)
(pendulum_fit.R:268,286) and rstan's chains (pendulum_fit.R:206).  Here: one process per GPU
(torch.distributed), a static contiguous split of the B items, NO collective on the data path --
each rank evaluates its slice with its own handle; only the 5 doubles per item of results are
gathered at the end (all_gather over NCCL on GPUs, gloo in the CPU tests).
"""
from __future__ import annotations

import numpy as np


def shard_bounds(total: int, rank: int, world: int):
    """Contiguous split of `total` items; the first total % world ranks get one extra."""
    base, rem = divmod(int(total), int(world))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def weighted_bounds(costs, rank: int, world: int):
    """Contiguous split of len(costs) items with about equal total cost per rank: item i goes to the rank whose share
    of the total holds the midpoint of its cumulative-cost interval."""
    costs = np.asarray(costs, dtype=np.float64)
    mid = np.cumsum(costs) - 0.5 * costs
    total = float(costs.sum())

    def cut(r):
        return 0 if r <= 0 else len(costs) if r >= world else int(np.searchsorted(mid, total * r / world, side="left"))
    return cut(rank), cut(rank + 1)


def _gather(parts, B, bounds, world, group):
    """all_gather of every rank's (lml, grad, info) slice; bounds[r] = (lo, hi) of rank r."""
    import torch
    import torch.distributed as dist
    lml, grad, info = parts
    width = max(1, max(hi - lo for lo, hi in bounds))
    rank = dist.get_rank(group)
    lo, hi = bounds[rank]
    mine = np.zeros((width, 5))
    mine[:hi - lo, 0] = lml
    mine[:hi - lo, 1:4] = grad
    mine[:hi - lo, 4] = info
    backend = dist.get_backend(group)
    device = torch.device("cuda", torch.cuda.current_device()) if backend == "nccl" else torch.device("cpu")
    t = torch.from_numpy(mine).to(device)
    out = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(out, t, group=group)
    full = np.zeros((B, 5))
    for r in range(world):
        a, b = bounds[r]
        full[a:b] = out[r].cpu().numpy()[:b - a]
    return full[:, 0].copy(), full[:, 1:4].copy(), full[:, 4].astype(np.int32)


def lml_grad_groups_sharded(xs, ys, theta, jitter=0.0, evaluator=None, group=None):
    """Per-group GPs of different sizes across the ranks of the default process group.

    xs, ys: lists of B 1-D arrays; theta (B, 3).  Each rank takes a contiguous range of groups holding about 1/world of
    the total sum of n_b^3 (the cost of a group's factorisation and inverse), not of the count, and evaluates it with
    one ragged call.  evaluator(xs, ys, theta_slice, jitter) -> (lml, grad, info) defaults to the GPU handle of this
    rank's device.  Returns the full (lml[B], grad[B,3], info[B]) on every rank.
    """
    import torch
    import torch.distributed as dist
    theta = np.ascontiguousarray(theta, dtype=np.float64).reshape(-1, 3)
    B = theta.shape[0]
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    costs = [float(np.asarray(v).size) ** 3 for v in xs]
    bounds = [weighted_bounds(costs, r, world) for r in range(world)]
    lo, hi = bounds[rank]
    if evaluator is None:
        from . import capi
        dev = torch.cuda.current_device() if torch.cuda.is_available() else 0
        h = capi.default_handle(dev)
        evaluator = lambda a, b, t, j: h.lml_grad_ragged(a, b, t, j)  # noqa: E731
    if hi > lo:
        parts = evaluator(list(xs[lo:hi]), list(ys[lo:hi]), theta[lo:hi], jitter)
    else:
        parts = np.empty(0), np.empty((0, 3)), np.empty(0, dtype=np.int32)
    if world == 1:
        return parts
    return _gather(parts, B, bounds, world, group)


def lml_grad_draws_sharded(x, y, theta, jitter=0.0, evaluator=None, group=None):
    """Evaluate B = len(theta) independent items across the ranks of the default process group.

    x, y: shared (n,) or per item (B, n).  evaluator(x, y, theta_slice, jitter) -> (lml, grad, info)
    defaults to the GPU handle of this rank's device; tests inject a CPU evaluator to exercise the
    plumbing with the gloo backend.  Returns the full (lml[B], grad[B,3], info[B]) on every rank.
    """
    import torch
    import torch.distributed as dist
    theta = np.ascontiguousarray(theta, dtype=np.float64)
    B = theta.shape[0]
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    lo, hi = shard_bounds(B, rank, world)
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    xs = x[lo:hi] if x.ndim == 2 else x
    ys = y[lo:hi] if y.ndim == 2 else y
    if evaluator is None:
        from . import capi
        dev = torch.cuda.current_device() if torch.cuda.is_available() else 0
        h = capi.default_handle(dev)
        evaluator = lambda a, b, t, j: h.lml_grad_batched(a, b, t, j)  # noqa: E731
    if hi > lo:
        lml, grad, info = evaluator(xs, ys, theta[lo:hi], jitter)
    else:
        lml, grad, info = np.empty(0), np.empty((0, 3)), np.empty(0, dtype=np.int32)
    if world == 1:
        return lml, grad, info
    # fixed-size gather: pad every slice to the largest one
    width = (B + world - 1) // world
    mine = np.zeros((width, 5))
    mine[:hi - lo, 0] = lml
    mine[:hi - lo, 1:4] = grad
    mine[:hi - lo, 4] = info
    backend = dist.get_backend(group)
    device = torch.device("cuda", torch.cuda.current_device()) if backend == "nccl" else torch.device("cpu")
    t = torch.from_numpy(mine).to(device)
    out = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(out, t, group=group)
    full = np.zeros((B, 5))
    for r in range(world):
        a, b = shard_bounds(B, r, world)
        full[a:b] = out[r].cpu().numpy()[:b - a]
    return full[:, 0].copy(), full[:, 1:4].copy(), full[:, 4].astype(np.int32)
