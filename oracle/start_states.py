"""NumPy restatement of the start states of ``msat_apply_start_states`` (test oracle only), and of the rollout of
``oracle/rollout.py`` with start states applied after the initial reset and after every auto-reset.

Start-state contract (include/marl_sat_b200.h, word for word).
  - Env b is rewritten iff its state record has step == 0 and has_start[p] != 0, with p its problem index clamped
    into [0, num_problems) as msat_reset clamps it.  step == 0 is what msat_reset and an auto-reset leave (and
    msat_import_state given step 0); every env that did not restart has step >= 1.  Nothing is written for any
    other env, not even its observation row.
  - Key: K = split(reset_key, num_envs_global)[g] for the global env g = env_offset + b -- the key msat_env_keys
    and the fused step derive -- and (ka, kb) = split(K).  randint reads only kb (env:162); the perturbation word
    of variable v is u_v = threefry_2x32(ka, arange(n))[v] (randint's counter layout), so the flips are
    independent of the reference draw and cost the same ceil(n/2) Threefry blocks.
  - Assignment: bit v = (start bit v) XOR (u_v < flip_thr[p]); flip_thr = 0 reproduces the start exactly.
    A flip probability q in [0, 1] is quantised on the host as flip_thr = min(round(q * 2^32), 2^32 - 1), so
    every bit flips with probability flip_thr / 2^32: q = 1 misses a flip with probability 2^-32.
  - State: clause status, num_unsatisfied and, on an MSAT_CLAUSES_INCREMENTAL plan, the 4-bit true-literal counts
    are recomputed from the bank record as msat_import_state does; step, problem index and done stay 0 / p / 0.
  - Outputs: obs (int32 or int8, following the plan) and the GNN inputs gnn_assignment int32[B,n] /
    gnn_clause_features float[B,m,3] are rewritten for the rewritten envs only, equal to msat_get_obs and
    msat_gnn_dynamic of the new state.  Any of them may be NULL.
  - Each result depends only on (reset_key, num_envs_global, g, p, the tables), so any sharding reproduces the
    single-device values.

The draws come from the KAT-pinned ``oracle.threefry``.
"""
from __future__ import annotations

from dataclasses import replace

import numpy as np

from . import threefry


def quantize_flip_prob(q) -> np.ndarray:
    """``flip_thr = min(round(q * 2^32), 2^32 - 1)`` in float64 (round half to even) -> int64."""
    return np.minimum(np.rint(np.asarray(q, np.float64) * 2.0 ** 32), float(2 ** 32 - 1)).astype(np.int64)


def pack_assignments(assign) -> np.ndarray:
    """Start words uint32 [P, ceil(n/32)]: bit v % 32 of word v // 32 is assign[:, v] != 0."""
    a = np.asarray(assign) != 0
    P, n = a.shape
    words = np.zeros((P, (n + 31) // 32), np.uint32)
    for v in range(n):
        words[:, v // 32] |= a[:, v].astype(np.uint32) << np.uint32(v % 32)
    return words


def flip_words(env_keys, n: int) -> np.ndarray:
    """u uint32 [B, n]: u[b, v] = threefry_2x32(ka, arange(n))[v] with (ka, kb) = split(env_keys[b])."""
    ka, _ = threefry.split_many(np.asarray(env_keys, np.uint32))
    npad = n + (n & 1)
    half = npad // 2
    lo_ctr = np.arange(half, dtype=np.uint32)[None, :]
    hi_ctr = (np.arange(half, dtype=np.uint32) + np.uint32(half))[None, :]
    if n & 1:
        hi_ctr = hi_ctr.copy()
        hi_ctr[0, -1] = 0                                            # the zero pad
    B = ka.shape[0]
    o0, o1 = threefry.threefry2x32(ka[:, 0:1], ka[:, 1:2], np.broadcast_to(lo_ctr, (B, half)),
                                   np.broadcast_to(hi_ctr, (B, half)))
    return np.concatenate([o0, o1], axis=1)[:, :n]


def start_assignments(start, flip_thr, problem_idx, env_keys) -> np.ndarray:
    """int32 [B, n]: start[p_b] XOR (u_b < flip_thr[p_b]) for the envs' problems p_b and reset keys."""
    start = np.asarray(start) != 0
    p = np.asarray(problem_idx, np.int64)
    u = flip_words(env_keys, start.shape[1]).astype(np.int64)
    thr = np.asarray(flip_thr, np.int64)[p][:, None]
    return (start[p] ^ (u < thr)).astype(np.int32)


def apply_start_states(env, state, obs, problem_idx, env_keys, starts):
    """msat_apply_start_states on an oracle state: ``starts`` = (start assignments [P, n], flip_thr [P], has_start [P]
    or None); ``problem_idx`` [B] and ``env_keys`` [B, 2] (= split(reset_key, Bg)[g]) of every env.  Returns
    ``(state, obs[B, A, D])`` with the selected rows rewritten."""
    start, thr, has = starts
    P = np.asarray(start).shape[0]
    p = np.clip(np.asarray(problem_idx, np.int64), 0, P - 1)
    has = np.ones(P, bool) if has is None else np.asarray(has) != 0
    sel = (np.asarray(state.step) == 0) & has[p]
    if not sel.any():
        return state, obs
    assign = state.variable_assignments.copy()
    assign[sel] = start_assignments(start, thr, p[sel], np.asarray(env_keys)[sel])
    status, num_unsat = env.calculate_satisfaction(assign, state.clauses)
    new = replace(state, variable_assignments=assign, clauses_satisfied_status=status, num_unsatisfied=num_unsat)
    obs = np.where(sel[:, None, None], env.get_obs_array(new), obs)
    return new, obs


def rollout_T(env, problems_clauses, key0, actions, starts):
    """``oracle.rollout.rollout_T`` (T steps from the runner's initial reset, actions from a table) with
    ``apply_start_states`` after the initial reset and after every step, on that call's env keys (the
    msat_apply_start_states call that follows msat_reset / each auto-resetting step).  ``starts`` = (assignments
    [P, n], flip_thr [P], has_start [P] | None).  Returns ``(transition, final)`` with the pre-step ``local_obs`` /
    GNN inputs, the pre-reset reward / done / info and the per-step ``act_key``; ``final`` holds state, obs, rng and
    the envs' problem indices."""
    from .features import state_to_gnn_input
    from .rollout import env_step_with_autoreset, initial_reset_inputs, rollout_keys
    T, B = actions.shape[0], actions.shape[1]
    P = problems_clauses.shape[0]
    rng, idx0, keys0 = initial_reset_inputs(np.asarray(key0, np.uint32), B, P)
    obs, state = env.reset(problems_clauses[idx0], keys0)
    obs = np.stack([obs[a] for a in env.agents], axis=1)
    pidx = np.asarray(idx0, np.int64)
    state, obs = apply_start_states(env, state, obs, pidx, keys0, starts)
    tr = {k: [] for k in ("local_obs", "gs_assignment", "gs_clause_features", "reward", "global_done", "info_solved",
                          "info_num_unsatisfied", "info_episode_step", "act_key")}
    for t in range(T):
        gs = state_to_gnn_input(env, state)
        tr["local_obs"].append(obs)
        tr["gs_assignment"].append(gs["assignment"])
        tr["gs_clause_features"].append(gs["clause_features"])
        ks = rollout_keys(rng, B, P)
        rng = ks["rng"]
        tr["act_key"].append(ks["act_key"])
        obs, state, reward, done_all, infos = env_step_with_autoreset(
            env, state, actions[t], problems_clauses, ks["new_problem_indices"], ks["reset_keys"])
        pidx = np.where(done_all, ks["new_problem_indices"], pidx)
        state, obs = apply_start_states(env, state, obs, pidx, ks["reset_keys"], starts)
        tr["reward"].append(reward)
        tr["global_done"].append(done_all)
        for k in ("solved", "num_unsatisfied", "episode_step"):
            tr["info_" + k].append(infos[k])
    return {k: np.stack(v) for k, v in tr.items()}, {"obs": obs, "state": state, "rng": rng, "problem_idx": pidx}
