"""NumPy restatement of the on-device action draw ``msat_sample_actions`` (test oracle only).

The reference draws each rollout step's joint action with ``rng, act_key = split(rng); action =
pi.sample(seed=act_key)`` (learner:397-403): a distrax 0.1.5 ``Categorical`` over the actor's logits, sampled
with JAX 0.4.29's ``jax.random.categorical``.  The contract, as stated in include/marl_sat_b200.h:

* logits float32 ``[rows, C]`` form one global table; element ``e = row * C + c`` of ``N = rows * C``.
* ``act_key = split(rng)[1]``.
* ``bits_e = threefry_2x32(act_key, arange(N))[e]``;
  ``f_e = bitcast_f32((bits_e >> 9) | 0x3F800000) - 1``;
  ``u_e = max(FLT_MIN, f_e * (1 - FLT_MIN) + FLT_MIN)`` in float32 (``uniform(minval=finfo.tiny, maxval=1)``);
  ``g_e = -log(-log(u_e))`` (``jax.random.gumbel``).
* Per row ``z = log_softmax(l)``: ``M = max l``, ``z_c = (l_c - M) - log(sum_c exp(l_c - M))``; ``action`` is the
  smallest ``c`` maximising ``g_c + z_c`` (``jnp.argmax``) and ``log_prob = z_action``.
* A row with a NaN or +inf logit, or with every logit -inf, gets ``action = -1`` and ``log_prob = -inf``.

The categorical / gumbel / uniform and ``Categorical`` details are restated from the published sources: JAX is not
available here to confirm them.  The Threefry bits are pinned by known-answer tests (tests/test_threefry_kat.py)
and the key by the reference fixtures' ``act_keys``.  ``bits``, ``f`` and ``u`` are exact here; ``g`` and ``z`` are
computed in float64, so the device's float32 values differ in the last bits and ``margin`` tells near-ties apart.
"""
from __future__ import annotations

import numpy as np

from . import threefry

_TINY = np.float32(np.finfo(np.float32).tiny)


def act_key(rng) -> np.ndarray:
    """``split(rng)[1]``: the sampling key of the rollout step that advances ``rng`` (learner:397)."""
    return threefry.split(np.asarray(rng, np.uint32))[1]


def uniform_bits(key, n: int) -> tuple[np.ndarray, np.ndarray]:
    """The random bits of ``n`` elements and their float32 uniforms ``u`` in ``[FLT_MIN, 1)``."""
    bits = threefry.random_bits32(np.asarray(key, np.uint32), n)
    f = ((bits >> np.uint32(9)) | np.uint32(0x3F800000)).view(np.float32) - np.float32(1.0)
    u = np.maximum(_TINY, f * (np.float32(1.0) - _TINY) + _TINY).astype(np.float32)
    return bits, u


def gumbel(u: np.ndarray) -> np.ndarray:
    """``-log(-log(u))`` in float64."""
    return -np.log(-np.log(u.astype(np.float64)))


def categorical(key, logits) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Draw from every row of ``logits`` (``[..., C]``, the whole global table) with ``key`` (the act_key).

    Returns ``(action int32, log_prob float64, margin float64)`` of shape ``logits.shape[:-1]``; ``margin`` is the
    best score minus the second best (``inf`` for one class or a single finite score, and for invalid rows)."""
    l32 = np.asarray(logits, np.float32)
    shape, C = l32.shape[:-1], l32.shape[-1]
    l = l32.reshape(-1, C).astype(np.float64)
    _, u = uniform_bits(key, l.size)
    g = gumbel(u).reshape(l.shape)
    invalid = np.isnan(l).any(1) | np.isposinf(l).any(1) | np.isneginf(l).all(1)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        M = np.where(invalid, 0.0, l.max(1))
        shifted = l - M[:, None]
        z = shifted - np.log(np.exp(shifted).sum(1))[:, None]
        score = np.where(invalid[:, None], 0.0, g + z)
    action = score.argmax(1)
    rows = np.arange(l.shape[0])
    best = score[rows, action]
    if C > 1:
        second = np.partition(score, C - 2, axis=1)[:, C - 2]
        with np.errstate(invalid="ignore"):
            margin = np.where(np.isfinite(second), best - second, np.inf)
    else:
        margin = np.full(l.shape[0], np.inf)
    log_prob = z[rows, action]
    action = np.where(invalid, -1, action).astype(np.int32)
    log_prob = np.where(invalid, -np.inf, log_prob)
    margin = np.where(invalid, np.inf, margin)
    return action.reshape(shape), log_prob.reshape(shape), margin.reshape(shape)
