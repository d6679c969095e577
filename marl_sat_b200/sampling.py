"""On-device action draw from the rollout's act_key (``msat_sample_actions``).

The reference draws each rollout step's joint action with ``rng, act_key = split(rng); action =
pi.sample(seed=act_key)`` (learner:397-403).  ``sample_actions`` is that draw for a float32 logits table: the
Gumbel-max sample of ``jax.random.categorical`` over the log-softmax of each row, with the Threefry bits of the
whole global table, so every sharding of the rows reproduces the single-device draw bit for bit.  The contract
(bits, uniforms, Gumbel values, tie rule, invalid rows) is spelled out in ``include/marl_sat_b200.h``;
``VecSATEnv.sample_actions`` binds it to a rollout's key chain and shard.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from . import _lib
from .env import ArrayLike, _ptr, _stream_ptr, as_u32_tensor


def _check_out(t: torch.Tensor, name: str, dtype: torch.dtype, shape, device: torch.device) -> None:
    if not isinstance(t, torch.Tensor) or t.dtype != dtype or tuple(t.shape) != tuple(shape) or t.device != device \
            or not t.is_contiguous():
        raise ValueError(f"{name} must be a contiguous {dtype} tensor of shape {tuple(shape)} on {device}")


def sample_actions(logits: torch.Tensor, rng: ArrayLike, num_rows_global: Optional[int] = None, row_offset: int = 0,
                   actions: Optional[torch.Tensor] = None,
                   log_prob: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Draw one class per row of ``logits`` (float32 ``[..., C]``, contiguous, on a CUDA device) with
    ``act_key = split(rng)[1]``, where ``rng`` (uint32 ``[2]``, a device tensor for graph capture) is the rollout rng
    the next step will advance.  The rows are rows ``[row_offset, row_offset + rows)`` of a global table of
    ``num_rows_global`` rows (default: this table alone).  Returns ``(actions int32, log_prob float32)`` of shape
    ``logits.shape[:-1]``: the drawn class and its log-softmax value, or ``-1`` / ``-inf`` for a row with a NaN or
    +inf logit or with every logit -inf.  ``actions`` / ``log_prob`` may be given preallocated (then the call
    allocates nothing and can be captured in a CUDA graph).  Enqueue only; there is no CPU path."""
    if not isinstance(logits, torch.Tensor) or logits.dtype != torch.float32:
        raise ValueError("logits must be a float32 tensor")
    if logits.dim() < 1 or logits.shape[-1] < 1:
        raise ValueError(f"logits must be [..., C] with C >= 1, got {tuple(logits.shape)}")
    if not logits.is_contiguous():
        raise ValueError("logits must be contiguous")
    dev = logits.device
    shape, C = tuple(logits.shape[:-1]), int(logits.shape[-1])
    rows = logits.numel() // C
    num_rows_global = rows if num_rows_global is None else int(num_rows_global)
    row_offset = int(row_offset)
    if row_offset < 0 or row_offset + rows > num_rows_global:
        raise ValueError(f"rows [{row_offset}, {row_offset + rows}) lie outside the global table of "
                         f"{num_rows_global} rows")
    if num_rows_global * C >= 2 ** 32 - 1:
        raise ValueError(f"the global table has {num_rows_global * C} elements; at most 2**32 - 2 are supported")
    if dev.type != "cuda":
        raise ValueError("logits must be on a CUDA device: sample_actions has no CPU path")
    rng =as_u32_tensor(rng, dev).reshape(-1)
    if rng.numel() != 2:
        raise ValueError("rng must hold one uint32[2] key")
    if actions is None:
        actions = torch.empty(shape, dtype=torch.int32, device=dev)
    _check_out(actions, "actions", torch.int32, shape, dev)
    if log_prob is None:
        log_prob = torch.empty(shape, dtype=torch.float32, device=dev)
    _check_out(log_prob, "log_prob", torch.float32, shape, dev)
    _lib.check(_lib.load().msat_sample_actions(_ptr(logits), num_rows_global, row_offset, rows, C, _ptr(rng),
                                               _ptr(actions), _ptr(log_prob), _stream_ptr(dev)),
               "msat_sample_actions")
    return actions, log_prob
