"""Sharding across the GPUs of one box, following the path's natural parallelism
(SURVEY.md 8e): one process per GPU, ``torch.distributed`` for the plumbing.

* independent problems (seeds, lambda1 / mu grids, bootstrap replicates): problem ``p`` goes
  to rank ``p mod G``; no communication on the data path, one gather of the results;
* large-n scores (logistic ``DagmaLinear``, ``DagmaNonlinear``): contiguous row shards of X,
  replicated parameters, ONE sum all-reduce of the d x d (or parameter-sized) gradient per
  inner iteration -- every rank then performs the identical update, so no broadcast.

The helpers take a ``solver`` callable so that the host logic (index arithmetic, gather and
re-ordering, reduction protocol) is testable with the gloo backend on CPU.
"""
from __future__ import annotations

import typing

import numpy as np
import torch
import torch.distributed as dist


def world(group=None) -> typing.Tuple[int, int]:
    if not (dist.is_available() and dist.is_initialized()):
        return 0, 1
    return dist.get_rank(group), dist.get_world_size(group)


def problem_shard(n_problems: int, rank: int, world_size: int) -> np.ndarray:
    """indices of the problems owned by ``rank`` (round robin: p mod G)."""
    return np.arange(rank, n_problems, world_size)


def row_shard(n: int, rank: int, world_size: int) -> slice:
    """contiguous rows of X owned by ``rank`` (sizes differ by at most one)."""
    base, rem = divmod(n, world_size)
    lo = rank * base + min(rank, rem)
    return slice(lo, lo + base + (1 if rank < rem else 0))


def allreduce_sum_(t: torch.Tensor, group=None) -> torch.Tensor:
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t


def gather_problems(local: torch.Tensor, n_problems: int, group=None) -> torch.Tensor:
    """Inverse of ``problem_shard``: every rank gets the [n_problems, ...] tensor in problem order."""
    rank, ws = world(group)
    if ws == 1:
        return local
    per = (n_problems + ws - 1) // ws
    pad = torch.zeros((per,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    pad[:local.shape[0]] = local
    parts = [torch.empty_like(pad) for _ in range(ws)]
    dist.all_gather(parts, pad, group=group)
    out = torch.empty((n_problems,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    for r in range(ws):
        idx = problem_shard(n_problems, r, ws)
        out[torch.as_tensor(idx, device=local.device)] = parts[r][:len(idx)]
    return out


def fit_batch_sharded(X=None, lambda1=0.03, *, cov=None, group=None, solver=None, device=None, **fit_kw):
    """``fit_batch`` with the problems split round-robin over the ranks of ``group``.

    Every rank passes the FULL problem list (host arrays) and receives the full thresholded
    ``W_est`` [n_problems, d, d] as numpy; each rank only stages and solves its own share."""
    rank, ws = world(group)
    src = X if X is not None else cov
    n_problems = len(src)
    idx = problem_shard(n_problems, rank, ws)
    lam = np.broadcast_to(np.asarray(lambda1, dtype=np.float64), (n_problems,))[idx]
    if solver is None:
        from .linear import fit_batch as solver          # the B200 path
    kw = dict(fit_kw)
    if isinstance(kw.get("trek_reg"), (list, tuple)):     # one regulariser per problem: it travels with its problem
        treks = kw["trek_reg"]
        if len(treks) != n_problems:
            raise ValueError(f"fit_batch_sharded: trek_reg has {len(treks)} entries for {n_problems} problems")
        kw["trek_reg"] = [treks[i] for i in idx]
    if device is not None:
        kw["device"] = device
    local_in = np.asarray(src)[idx] if not isinstance(src, torch.Tensor) else src[torch.as_tensor(idx)]
    if len(idx) == 0:                     # fewer problems than ranks: an empty share still joins the gather
        d = int(np.shape(src)[-1])
        W_local = np.zeros((0, d, d))
    else:
        W_local = solver(local_in, lam, **kw) if X is not None else solver(None, lam, cov=local_in, **kw)
    W_local = torch.as_tensor(np.ascontiguousarray(W_local))
    if ws > 1 and dist.get_backend(group) == "nccl":
        W_local = W_local.cuda()
    return gather_problems(W_local, n_problems, group).cpu().numpy()
