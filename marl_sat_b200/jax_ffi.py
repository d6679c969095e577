"""JAX side of the XLA FFI custom-call layer (``csrc/xla_ffi_shim.cc``): registration of the handlers and
``jax.ffi.ffi_call`` wrappers with the shapes of the reference's call sites
(``src/learners/mappo_gnn_sat_learner.py:418,435``, ``src/runners/mappo_runner.py:137``).

Needs JAX >= 0.4.38 (public ``jax.ffi``) -- NOT available in this image (SURVEY.md F2), so this module is
import-guarded, never imported by the package itself, and exercised only where JAX exists.  The reference pins
``jax==0.4.29``; its PRNG layout (``jax_threefry_partitionable=False``) is what the kernels reproduce, so a
newer JAX must run with ``jax.config.update("jax_threefry_partitionable", False)``.

Build the shim first: ``python marl_sat_b200/build.py --ffi`` (uses ``jax.ffi.include_dir()``).
"""
from __future__ import annotations

import ctypes
from pathlib import Path

import numpy as np

try:                                    # pragma: no cover - JAX is absent from the build image
    import jax
    import jax.numpy as jnp
    from jax import ffi as jffi
except Exception as e:                  # pragma: no cover
    raise ImportError("marl_sat_b200.jax_ffi needs JAX >= 0.4.38 (jax.ffi); the torch/ctypes host layer "
                      "(marl_sat_b200.SATEnv, VecSATEnv, ...) works without it") from e

SHIM_PATH = Path(__file__).resolve().parent / "csrc" / "libmarlsat_b200_xla.so"

# handler symbol -> FFI target name
TARGETS = {
    "MsatCompileBank": "msat_compile_bank", "MsatReset": "msat_reset", "MsatImportState": "msat_import_state",
    "MsatStep": "msat_step",
    "MsatRolloutSteps": "msat_rollout_steps", "MsatRolloutStepsGnn": "msat_rollout_steps_gnn",
    "MsatGetObs": "msat_get_obs", "MsatExportState": "msat_export_state", "MsatRngChain": "msat_rng_chain",
    "MsatRngSplit2": "msat_rng_split2", "MsatEnvKeys": "msat_env_keys",
    "MsatEnvKeysWeighted": "msat_env_keys_weighted", "MsatProblemStats": "msat_problem_stats", "MsatGae": "msat_gae",
    "MsatAdvStats": "msat_adv_stats", "MsatAdvNormalize": "msat_adv_normalize", "MsatGnnStatic": "msat_gnn_static",
    "MsatGnnDynamic": "msat_gnn_dynamic", "MsatRolloutMetrics": "msat_rollout_metrics",
    "MsatFlipGains": "msat_flip_gains", "MsatEvalTrack": "msat_eval_track", "MsatWalksat": "msat_walksat",
}
_registered = False


def register() -> None:
    """``jax.ffi.register_ffi_target`` for every handler of the shim (platform "CUDA"), once per process."""
    global _registered
    if _registered:
        return
    if not SHIM_PATH.exists():
        raise ImportError(f"{SHIM_PATH} is missing: build it with `python marl_sat_b200/build.py --ffi`")
    lib = ctypes.CDLL(str(SHIM_PATH))
    for symbol, target in TARGETS.items():
        jffi.register_ffi_target(target, jffi.pycapsule(getattr(lib, symbol)), platform="CUDA")
    _registered = True


def _sds(shape, dtype):
    return jax.ShapeDtypeStruct(tuple(int(x) for x in shape), dtype)


def reset(plan_handle: int, dims, bank, num_problems: int, problem_idx, keys):
    """``jax.vmap(env.reset)(clauses[problem_idx], keys)`` (env:158-181; runner:137) -> ``(state, obs)``."""
    register()
    B = problem_idx.shape[0]
    call = jffi.ffi_call("msat_reset", (_sds((B, dims.state_words), jnp.uint32), _sds((B, dims.A, dims.D), jnp.int32)))
    return call(bank, problem_idx, keys, plan=np.int64(plan_handle), num_problems=np.int64(num_problems))


def import_state(plan_handle: int, dims, bank, num_problems: int, problem_idx, variable_assignments, step=None,
                 done=None):
    """Inverse of ``MsatExportState``: packed states from reference-shaped ``SATState`` leaves (env:13-24), e.g. a
    reference ``reset``'s, a checkpoint's or an edited assignment -> ``(state, obs)``.  ``variable_assignments``
    [B, n] (0 / 1), ``step`` [B] (default 0, kept as given), ``done`` [B] or [B, A] (default False)."""
    register()
    B = problem_idx.shape[0]
    step = jnp.zeros((B,), jnp.int32) if step is None else jnp.asarray(step, jnp.int32)
    done = jnp.zeros((B,), jnp.uint8) if done is None else jnp.asarray(done)
    if done.ndim == 2:
        done = done[:, 0]
    call = jffi.ffi_call("msat_import_state", (_sds((B, dims.state_words), jnp.uint32),
                                               _sds((B, dims.A, dims.D), jnp.int32)))
    return call(bank, jnp.asarray(problem_idx, jnp.int32), jnp.asarray(variable_assignments, jnp.int32), step,
                done.astype(jnp.uint8), plan=np.int64(plan_handle), num_problems=np.int64(num_problems))


def walksat(plan_handle: int, bank, num_problems: int, state, keys, max_flips: int, noise: float = 0.5,
            flip_offset: int = 0):
    """WalkSAT/SKC on packed env states (``msat_walksat``; contract in include/marl_sat_b200.h).  ``state`` is
    donated (searched in place); ``keys`` uint32 [B, 2].  Returns ``(state, solved uint8[B], flips int32[B])``."""
    register()
    B = state.shape[0]
    call = jffi.ffi_call("msat_walksat", (_sds(state.shape, jnp.uint32), _sds((B,), jnp.uint8), _sds((B,), jnp.int32)),
                         input_output_aliases={1: 0})
    return call(bank, state, jnp.asarray(keys, jnp.uint32), plan=np.int64(plan_handle),
                num_problems=np.int64(num_problems), max_flips=np.int64(max_flips), flip_offset=np.int64(flip_offset),
                noise=np.float64(noise))


def rollout_steps(plan_handle: int, dims, bank, num_problems: int, state, actions, rng, num_envs_global=None,
                  env_offset: int = 0, emit_every_step: bool = False, reward_cols: int = 1, done_cols: int = 1):
    """The env half of ``_env_step`` (learner:397-464) for K = ``actions.shape[0]`` steps in one custom call.
    ``state`` is donated (updated in place).  Returns ``(state, chain, obs, reward, done, solved,
    num_unsatisfied, episode_step)``; ``chain[0:2]`` is the advanced rng."""
    register()
    K, B = actions.shape[0], actions.shape[1]
    lead = (K, B) if emit_every_step else (B,)
    out = (_sds(state.shape, jnp.uint32), _sds((10,), jnp.uint32), _sds(lead + (dims.A, dims.D), jnp.int32),
           _sds((K, B, reward_cols), jnp.float32), _sds((K, B, done_cols), jnp.uint8), _sds((K, B), jnp.uint8),
           _sds((K, B), jnp.int32), _sds((K, B), jnp.int32))
    call = jffi.ffi_call("msat_rollout_steps", out, input_output_aliases={1: 0})
    return call(bank, state, actions, rng, plan=np.int64(plan_handle), num_problems=np.int64(num_problems),
                num_steps=np.int64(K), num_envs_global=np.int64(num_envs_global or B), env_offset=np.int64(env_offset),
                emit_every_step=np.int64(1 if emit_every_step else 0))


def env_keys_weighted(prob_key, reset_key, cum_weights, num_envs_local: int, num_envs_global=None,
                      env_offset: int = 0):
    """Per-env problem indices drawn with the weights whose inclusive prefix sums are ``cum_weights`` (int64 [P]) and
    the reset keys of ``msat_env_keys``, for the shard ``[env_offset, env_offset + num_envs_local)`` -> ``(idx, keys)``.
    The draw contract is in include/marl_sat_b200.h; int64 buffers need ``jax_enable_x64``."""
    register()
    B = int(num_envs_local)
    call = jffi.ffi_call("msat_env_keys_weighted", (_sds((B,), jnp.int32), _sds((B, 2), jnp.uint32)))
    return call(prob_key, reset_key, jnp.asarray(cum_weights, jnp.int64),
                num_envs_global=np.int64(num_envs_global or B), env_offset=np.int64(env_offset))


def problem_stats(problem_idx, done, solved, num_unsatisfied, episode_step, num_problems: int, stats=None):
    """int64 ``[P, 4]`` per-problem statistics of a dense ``[T, B]`` rollout (``msat_problem_stats``), added to
    ``stats`` (default zeros).  Needs ``jax_enable_x64``."""
    register()
    P = int(num_problems)
    stats = jnp.zeros((P, 4), jnp.int64) if stats is None else stats
    call = jffi.ffi_call("msat_problem_stats", _sds((P, 4), jnp.int64), input_output_aliases={5: 0})
    return call(jnp.asarray(problem_idx, jnp.int32), done.astype(jnp.uint8), solved.astype(jnp.uint8),
                jnp.asarray(num_unsatisfied, jnp.int32), jnp.asarray(episode_step, jnp.int32), stats)


def calculate_gae(reward, done, value, last_val, gamma: float, gae_lambda: float):
    """``_calculate_gae`` (learner:504-528) + the statistics of the normalisation (learner:530-531):
    ``(advantages, targets, stats)`` with ``stats = (count, sum, sum of squares)`` in float64."""
    register()
    T, B = value.shape
    out = (_sds((T, B), jnp.float32), _sds((T, B), jnp.float32), _sds((3,), jnp.float64))
    call = jffi.ffi_call("msat_gae", out, input_output_aliases={4: 2})
    return call(reward, done.astype(jnp.uint8), value, last_val, jnp.zeros((3,), jnp.float64),
                gamma=np.float64(gamma), gae_lambda=np.float64(gae_lambda))


def normalize_advantages(adv, stats):
    """learner:530-532 with (optionally ``jax.lax.psum``-reduced) statistics; ``adv`` is donated."""
    register()
    call = jffi.ffi_call("msat_adv_normalize", _sds(adv.shape, jnp.float32), input_output_aliases={0: 0})
    return call(adv, stats)
