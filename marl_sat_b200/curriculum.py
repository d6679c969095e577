"""Curricula over the formula bank: per-problem rollout statistics and weighted problem draws for auto-reset.

``problem_stats`` reduces a ``[T, B]`` rollout to int64 ``[P, 4]`` per-problem counters on the device
(``msat_problem_stats``); ``problem_weights`` quantises a weight vector into the integer form the weighted draw reads
(``msat_env_keys_weighted``); ``unsolved_weights`` is one priority rule built from the statistics.
``VecSATEnv.set_problem_weights`` installs the weights for auto-reset.  Together they allow curricula such as "only
the formulas WalkSAT solved" or "weight each formula by its unsolved rate".  The draw keeps the shard invariance of
the uniform one (DESIGN.md section 7): each env's index depends only on the rollout rng, its global env index, the
global batch size and the weights.
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from . import _lib
from .env import ArrayLike, _ptr, _stream_ptr

STATS_COLUMNS = ("finished", "solved", "sum_num_unsatisfied", "sum_steps_solved")
_QMAX = float(2 ** 32 - 1)


def problem_weights(weights: ArrayLike, num_problems: Optional[int] = None) -> torch.Tensor:
    """Quantise non-negative problem weights to int64 ``[P]`` (host): ``q = round(w / max(w) * (2^32 - 1))`` in
    float64 (round half to even), so the largest weight becomes 2^32 - 1 and a weight of 0 stays 0.  Raises
    ``ValueError`` for a shape other than ``[P]`` (``[num_problems]`` when given), a NaN, infinite or negative value,
    or all values zero."""
    w = weights.detach().cpu().numpy() if isinstance(weights, torch.Tensor) else np.asarray(weights)
    if w.ndim != 1 or w.shape[0] == 0 or (num_problems is not None and w.shape[0] != int(num_problems)):
        want = f"[{int(num_problems)}]" if num_problems is not None else "[P] with P >= 1"
        raise ValueError(f"problem weights must have shape {want}, got {tuple(w.shape)}")
    if not (w.dtype == np.bool_ or np.issubdtype(w.dtype, np.integer) or np.issubdtype(w.dtype, np.floating)):
        raise ValueError(f"problem weights must be real numbers, got dtype {w.dtype}")
    w = w.astype(np.float64)
    if not np.isfinite(w).all():
        raise ValueError("problem weights must be finite (no NaN or infinity)")
    if (w < 0).any():
        raise ValueError("problem weights must be non-negative")
    top = w.max()
    if top == 0:
        raise ValueError("problem weights are all zero: no problem could be drawn")
    return torch.from_numpy(np.rint(w / top * _QMAX).astype(np.int64))


def unsolved_weights(stats: torch.Tensor, floor: float = 0.1) -> torch.Tensor:
    """Priority by unsolved rate from ``problem_stats`` totals: ``max(1 - solved / finished, floor)`` per problem,
    and 1 for a problem without a finished episode (float64 ``[P]``, on the device of ``stats``)."""
    if stats.dim() != 2 or stats.shape[1] != 4:
        raise ValueError(f"stats must be [P, 4] (problem_stats), got {tuple(stats.shape)}")
    finished, solved = stats[:, 0].to(torch.float64), stats[:, 1].to(torch.float64)
    rate = (1.0 - solved / finished.clamp_min(1.0)).clamp_min(float(floor))
    return torch.where(finished > 0, rate, torch.ones_like(rate))


def _dense_u8(t: torch.Tensor) -> torch.Tensor:
    return (t.view(torch.uint8) if t.dtype == torch.bool else t).contiguous()


def problem_stats(problem_idx: torch.Tensor, done: torch.Tensor, solved: torch.Tensor, num_unsatisfied: torch.Tensor,
                  episode_step: torch.Tensor, num_problems: int, stats: Optional[torch.Tensor] = None,
                  group=None) -> torch.Tensor:
    """Per-problem statistics of a ``[T, B]`` rollout: int64 ``[P, 4]`` with, for every row that ends an episode
    (``done``), one episode added to its problem's row: #finished, #solved at finish, sum of ``num_unsatisfied`` at
    finish, sum of ``episode_step`` over the episodes solved at finish (``STATS_COLUMNS``; the order of
    ``rollout_metric_sums`` 1..4).  ``problem_idx`` int32 ``[T, B]`` may be any strided view -- e.g. the problem-index
    word of a ``RolloutBuffer.state`` (``RolloutBuffer.problem_stats``) -- and is read without a copy; indices are
    clamped into ``[0, P)``.  With ``torch.distributed`` initialised this rollout's counters are summed over the
    ranks of ``group``.  When ``stats`` (int64 ``[P, 4]`` running totals on the same device) is given the reduced
    counters are added to it and it is returned; the totals themselves are never all-reduced."""
    from .gae import allreduce_stats
    lib = _lib.load()
    P = int(num_problems)
    if P <= 0:
        raise ValueError(f"num_problems must be positive, got {P}")
    if done.dim() == 3:                        # RolloutBuffer.done [T, B, 1]: the global done column
        done = done[:, :, -1]
    if problem_idx.dim() != 2:
        raise ValueError(f"problem_idx must be [T, B], got {tuple(problem_idx.shape)}")
    T, B = problem_idx.shape
    dev = problem_idx.device
    if not problem_idx.is_cuda:
        raise RuntimeError("problem_stats needs CUDA tensors: there is no CPU fallback")
    if problem_idx.dtype != torch.int32:
        raise TypeError(f"problem_idx must be int32, got {problem_idx.dtype}")
    for name, t, dtypes in (("done", done, (torch.bool, torch.uint8)), ("solved", solved, (torch.bool, torch.uint8)),
                            ("num_unsatisfied", num_unsatisfied, (torch.int32,)),
                            ("episode_step", episode_step, (torch.int32,))):
        if tuple(t.shape) != (T, B) or t.dtype not in dtypes or t.device != dev:
            raise ValueError(f"{name} must be {'/'.join(str(d) for d in dtypes)} [{T}, {B}] on {dev}, "
                             f"got {t.dtype} {tuple(t.shape)} on {t.device}")
    if stats is not None and (tuple(stats.shape) != (P, 4) or stats.dtype != torch.int64 or stats.device != dev
                              or not stats.is_contiguous()):
        raise ValueError(f"stats must be a contiguous int64 [{P}, 4] tensor on {dev}")
    local = torch.zeros((P, 4), dtype=torch.int64, device=dev)
    _lib.check(lib.msat_problem_stats(_ptr(problem_idx), problem_idx.stride(0), problem_idx.stride(1),
                                      _ptr(_dense_u8(done)), _ptr(_dense_u8(solved)), _ptr(num_unsatisfied.contiguous()),
                                      _ptr(episode_step.contiguous()), T, B, P, _ptr(local), _stream_ptr(dev)),
               "msat_problem_stats")
    local = allreduce_stats(local, group)
    if stats is None:
        return local
    return stats.add_(local)
