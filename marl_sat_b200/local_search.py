"""Batched WalkSAT over env states (``msat_walksat``): a classical local-search solver next to the env.

``walksat`` runs WalkSAT/SKC (noise ``p``) on every env of a ``SATState`` and returns an ordinary ``SATState`` --
``get_obs``, the exported leaves, ``import_state``, checkpoints and ``evaluate_policy`` work on it unchanged.  Uses:
satisfying assignments for the formulas of a bank (the reference labels them with PySAT,
``src/utils/sat_solver.py``), a local-search baseline at the flip budget of an RL episode (``max_steps × A``
flips), and near-solution starts for ``SATEnv.import_state``.  The algorithm contract (clause choice by rank, break
counts, freebie / random walk / greedy) is spelled out in ``include/marl_sat_b200.h``.
"""
from __future__ import annotations

import math
from typing import NamedTuple

import torch

from . import _lib
from .env import ArrayLike, SATState, _ptr, _stream_ptr, as_u32_tensor

_MAX_I32 = 2 ** 31 - 1


class WalkSATResult(NamedTuple):
    state: SATState          # the searched states (a new packed tensor; the input state is not modified)
    solved: torch.Tensor     # bool [B]: num_unsatisfied == 0 after the search
    flips: torch.Tensor      # int32 [B]: flip iterations this call used


def walksat(state: SATState, keys: ArrayLike, max_flips: int, noise: float = 0.5,
            flip_offset: int = 0) -> WalkSATResult:
    """WalkSAT/SKC on a copy of ``state.packed``: per env at most ``max_flips`` iterations, stopping as soon as the
    env is solved.  ``keys`` uint32 ``[B, 2]`` (one Threefry key per env, required as in ``reset_from_bank``);
    ``noise`` in ``[0, 1]`` is the random-walk probability.  Iteration ``t`` draws its random bits with counter
    ``flip_offset + t``, so ``walksat(walksat(s, keys, F1).state, keys, F2, flip_offset=F1)`` equals
    ``walksat(s, keys, F1 + F2)`` bit for bit.  The step counter, done flag and problem index stay as they are.
    Enqueue only (no host synchronisation), so the call can be captured in a CUDA graph."""
    env = state.env
    dev = env._require_cuda()
    B = state.num_envs
    for name, val in (("max_flips", max_flips), ("flip_offset", flip_offset)):
        if isinstance(val, bool) or int(val) != val or val < 0:
            raise ValueError(f"{name} must be a non-negative integer, got {val!r}")
    max_flips, flip_offset = int(max_flips), int(flip_offset)
    if flip_offset + max_flips > _MAX_I32:
        raise ValueError(f"flip_offset + max_flips must be <= 2**31 - 1, got {flip_offset + max_flips}")
    noise = float(noise)
    if math.isnan(noise) or not 0.0 <= noise <= 1.0:
        raise ValueError(f"noise must lie in [0, 1], got {noise}")
    keys = as_u32_tensor(keys, dev)
    if not state.batched:
        keys = keys.reshape(-1, 2)
    if tuple(keys.shape) != (B, 2):
        raise ValueError(f"keys must be [{B}, 2] (one PRNG key per env), got {tuple(keys.shape)}")
    packed = state.packed.clone()
    solved = torch.empty(B, dtype=torch.uint8, device=dev)
    flips = torch.empty(B, dtype=torch.int32, device=dev)
    bank = state.bank
    _lib.check(env._lib.msat_walksat(bank.plan.handle, _ptr(bank.data), bank.num_problems, _ptr(packed), _ptr(keys),
                                     max_flips, flip_offset, noise, _ptr(solved), _ptr(flips), B, _stream_ptr(dev)),
               "msat_walksat")
    return WalkSATResult(SATState(env, bank, packed, state.batched), solved.bool(), flips)
