"""NumPy restatement of the curriculum primitives (test oracle only): the weighted problem draw of
``msat_env_keys_weighted`` and the per-problem statistics of ``msat_problem_stats``.

Weighted draw contract (include/marl_sat_b200.h, word for word).  For global env g out of Bg:
  - take the two 32-bit words randint already uses for that env: (k1, k2) = split(prob_key),
    hi = bits32_at(k1, Bg, g), lo = bits32_at(k2, Bg, g); let u = hi * 2^32 + lo;
  - cum_weights int64[P] holds inclusive prefix sums of non-negative integer weights; W = cum_weights[P-1];
  - if W <= 0 the index is the uniform draw, equal to what msat_env_keys returns;
  - otherwise r = floor(u * W / 2^64) (umulhi) and the index is the smallest p with cum_weights[p] > r;
  - the index is always in [0, P), also when the table is not monotone: the binary search is bounded;
  - reset_keys are identical to msat_env_keys' output.
Each draw depends only on (prob_key, Bg, g, cum_weights), so any sharding yields the single-device values.

The draws come from the KAT-pinned ``oracle.threefry``; ``umulhi`` is evaluated with Python integers (exact 128-bit
products).
"""
from __future__ import annotations

import numpy as np

from . import threefry


def weighted_randint(prob_key, num_envs: int, cum_weights) -> np.ndarray:
    """The weighted draw for all ``num_envs`` global envs -> int32 [num_envs]."""
    cum = [int(c) for c in np.asarray(cum_weights, np.int64)]
    P = len(cum)
    W = cum[-1]
    if W <= 0:
        return threefry.randint(prob_key, num_envs, 0, P)
    k1, k2 = threefry.split(prob_key)
    hi = threefry.random_bits32(k1, num_envs)
    lo = threefry.random_bits32(k2, num_envs)
    out = np.empty(num_envs, np.int32)
    for g in range(num_envs):
        u = (int(hi[g]) << 32) | int(lo[g])
        r = (u * W) >> 64                                   # umulhi(u, W)
        a, b = 0, P - 1                                     # bounded binary search: smallest p with cum[p] > r
        while a < b:
            mid = (a + b) >> 1
            if cum[mid] > r:
                b = mid
            else:
                a = mid + 1
        out[g] = a
    return out


def quantize_weights(weights) -> np.ndarray:
    """``q = round(w / max(w) * (2^32 - 1))`` in float64 (round half to even) -> int64 [P]."""
    w = np.asarray(weights, np.float64)
    return np.rint(w / w.max() * float(2 ** 32 - 1)).astype(np.int64)


def problem_stats(problem_idx, done, solved, num_unsatisfied, episode_step, num_problems: int) -> np.ndarray:
    """int64 [P, 4]: per finished episode (done[t, b]) of problem clamp(problem_idx[t, b], 0, P-1):
    #finished, #solved at finish, sum num_unsatisfied at finish, sum episode_step of solved-at-finish."""
    done = np.asarray(done).astype(bool)
    solved = np.asarray(solved).astype(bool) & done
    p = np.clip(np.asarray(problem_idx, np.int64), 0, num_problems - 1)
    stats = np.zeros((num_problems, 4), np.int64)
    np.add.at(stats[:, 0], p[done], 1)
    np.add.at(stats[:, 1], p[solved], 1)
    np.add.at(stats[:, 2], p[done], np.asarray(num_unsatisfied, np.int64)[done])
    np.add.at(stats[:, 3], p[solved], np.asarray(episode_step, np.int64)[solved])
    return stats


# --- the rollout of oracle/rollout.py with the weighted draw in place of randint ------------------------------------

def initial_reset_inputs(key, num_envs: int, cum_weights):
    """runner:289-295 with the weighted draw: ``key, _rng = split(key)``; ``_rng`` feeds both draws."""
    key, _rng = threefry.split(np.asarray(key, np.uint32))
    return key, weighted_randint(_rng, num_envs, cum_weights), threefry.split(_rng, num_envs)


def rollout_keys(rng, num_envs: int, cum_weights):
    """``oracle.rollout.rollout_keys`` with ``new_problem_indices`` from the weighted draw."""
    rng, act_key = threefry.split(rng)                       # learner:397
    rng, step_key = threefry.split(rng)                      # learner:416
    rng, prob_key, reset_key = threefry.split(rng, 3)        # learner:426
    return {"rng": rng, "act_key": act_key, "step_key": step_key, "prob_key": prob_key, "reset_key": reset_key,
            "new_problem_indices": weighted_randint(prob_key, num_envs, cum_weights),
            "reset_keys": threefry.split(reset_key, num_envs)}


def rollout_T(env, problems_clauses, key0, actions, cum_weights):
    """``oracle.rollout.rollout_T`` (T steps from the runner's initial reset, actions from a table) with every problem
    drawn by the weighted draw.  Returns ``(transition, final)`` with the pre-step ``local_obs`` / GNN inputs, the
    pre-reset reward / done / info and the per-step ``act_key``; ``final`` holds state, obs, rng and the initial
    problem indices."""
    from .features import state_to_gnn_input
    from .rollout import env_step_with_autoreset
    T, B = actions.shape[0], actions.shape[1]
    rng, idx0, keys0 = initial_reset_inputs(key0, B, cum_weights)
    obs, state = env.reset(problems_clauses[idx0], keys0)
    obs = np.stack([obs[a] for a in env.agents], axis=1)
    tr = {k: [] for k in ("local_obs", "gs_assignment", "gs_clause_features", "reward", "global_done", "info_solved",
                          "info_num_unsatisfied", "info_episode_step", "act_key")}
    for t in range(T):
        gs = state_to_gnn_input(env, state)
        tr["local_obs"].append(obs)
        tr["gs_assignment"].append(gs["assignment"])
        tr["gs_clause_features"].append(gs["clause_features"])
        ks = rollout_keys(rng, B, cum_weights)
        rng = ks["rng"]
        tr["act_key"].append(ks["act_key"])
        obs, state, reward, done_all, infos = env_step_with_autoreset(
            env, state, actions[t], problems_clauses, ks["new_problem_indices"], ks["reset_keys"])
        tr["reward"].append(reward)
        tr["global_done"].append(done_all)
        for k in ("solved", "num_unsatisfied", "episode_step"):
            tr["info_" + k].append(infos[k])
    return {k: np.stack(v) for k, v in tr.items()}, {"obs": obs, "state": state, "rng": rng, "problem_idx0": idx0}
