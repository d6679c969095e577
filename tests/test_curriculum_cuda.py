"""GPU tests of the curriculum primitives: the weighted problem draw (``msat_env_keys_weighted``,
``VecSATEnv.set_problem_weights``) and the per-problem statistics (``msat_problem_stats``, ``problem_stats``,
``RolloutBuffer.problem_stats``), against the NumPy oracle (``oracle/curriculum.py``) bit for bit."""
import os
import socket

import numpy as np
import pytest
import torch

from oracle import curriculum as ocur
from oracle import rollout as orollout
from oracle import threefry as otf
from oracle.features import state_to_gnn_input
from oracle.sat_env import SATEnvOracle
from tests.util import assert_state_equal, to_np

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")


def _msat():
    import marl_sat_b200 as M
    return M


def _weights(kind, P, seed):
    rng = np.random.default_rng(seed)
    if kind == "onehot":
        w = np.zeros(P)
        w[rng.integers(P)] = 1.0
    elif kind == "sparse":
        w = np.where(rng.random(P) < 0.05, rng.random(P) + 0.01, 0.0)
        w[rng.integers(P)] = 1.0
    elif kind == "uniform":
        w = np.ones(P)
    else:                                       # heavy-tailed: quantised values span 1 .. 2^32 - 1
        w = rng.pareto(0.3, P) + 1e-9
    return _msat().problem_weights(w)


def _u32(x):
    return _msat().env.as_u32_tensor(x, DEV)


def _derive(M, pk, rk, Bg, off, cnt, P, cum):
    idx = torch.empty(cnt, dtype=torch.int32, device=DEV)
    keys = torch.empty((cnt, 2), dtype=torch.int32, device=DEV)
    M.derive_env_keys(pk, rk, Bg, off, cnt, P, idx, keys, cum)
    return idx, keys


# ---------------------------------------------------------------------------------------------- weighted keys
@pytest.mark.parametrize("kind", ["onehot", "sparse", "uniform", "heavy"])
@pytest.mark.parametrize("P", [1, 7, 800, 65536])
def test_weighted_keys_match_the_oracle(P, kind):
    M = _msat()
    q = _weights(kind, P, seed=P + len(kind))
    cum_np = np.cumsum(q.numpy())
    cum = torch.from_numpy(cum_np).to(DEV)
    for Bg in (1, 33, 65536):
        pk, rk = otf.prng_key(Bg + P), otf.prng_key(7 * Bg + 1)
        idx, keys = _derive(M, _u32(pk), _u32(rk), Bg, 0, Bg, P, cum)
        exp = ocur.weighted_randint(pk, Bg, cum_np)
        assert np.array_equal(to_np(idx), exp), (P, kind, Bg)
        assert np.all(q.numpy()[to_np(idx)] > 0)
        u_idx, u_keys = _derive(M, _u32(pk), _u32(rk), Bg, 0, Bg, P, None)
        assert torch.equal(keys, u_keys)                                   # reset keys = msat_env_keys
        assert np.array_equal(M.env.u32_to_numpy(keys), otf.split(rk, Bg))


def test_weighted_keys_fallback_and_non_monotone_tables():
    M = _msat()
    Bg, P = 4097, 37
    pk, rk = otf.prng_key(5), otf.prng_key(6)
    for table in (np.zeros(P, np.int64), np.full(P, -9, np.int64),
                  np.random.default_rng(1).integers(-2 ** 40, 2 ** 40, P).astype(np.int64)):
        idx, _ = _derive(M, _u32(pk), _u32(rk), Bg, 0, Bg, P, torch.from_numpy(table).to(DEV))
        assert np.array_equal(to_np(idx), ocur.weighted_randint(pk, Bg, table))
        assert to_np(idx).min() >= 0 and to_np(idx).max() < P
        if table[-1] <= 0:
            assert np.array_equal(to_np(idx), otf.randint(pk, Bg, 0, P))


def test_weighted_keys_are_shard_invariant():
    M = _msat()
    Bg, P = 1001, 800
    q = _weights("heavy", P, 3)
    cum = torch.cumsum(q, 0).to(DEV)
    pk, rk = _u32(otf.prng_key(11)), _u32(otf.prng_key(12))
    full_idx, full_keys = _derive(M, pk, rk, Bg, 0, Bg, P, cum)
    for world in (2, 3, 8):
        parts = [_derive(M, pk, rk, Bg, *M.shard_range(Bg, world, r), P, cum) for r in range(world)]
        assert torch.equal(torch.cat([p[0] for p in parts]), full_idx), world
        assert torch.equal(torch.cat([p[1] for p in parts]), full_keys), world


# ---------------------------------------------------------------------------------------------- weighted rollouts
def _actions(rng, ref, T, B):
    if ref.action_mode == 0:
        return rng.integers(0, ref.max_vars_per_agent + 2, size=(T, B, ref.num_agents)).astype(np.int32)
    return rng.integers(0, 2, size=(T, B, ref.num_agents, ref.max_vars_per_agent)).astype(np.int32)


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("outputs", ["obs", "gnn"])
def test_weighted_rollout_matches_oracle_rollout_T(mode, outputs):
    M = _msat()
    n, m, B, P, T, max_steps = 20, 91, 64, 10, 9, 3
    from marl_sat_b200.synth import uniform_ksat
    problems = uniform_ksat(P, n, m, 3, seed=17)
    ref = SATEnvOracle(n, m, max_steps, action_mode=mode)
    env = M.SATEnv(n, m, max_steps, action_mode=mode, verbose=False)
    w = np.array([0.0, 1.0, 5.0, 0.0, 0.5, 2.0, 0.0, 0.0, 3.0, 1.0])
    q = M.problem_weights(w)
    key0 = otf.prng_key(42 + mode)
    acts = _actions(np.random.default_rng(mode), ref, T, B)
    tr, fin = ocur.rollout_T(ref, problems, key0, acts, np.cumsum(q.numpy()))
    gnn = outputs == "gnn"
    vec = M.VecSATEnv(env, torch.from_numpy(problems), B, key0, emit_obs=not gnn, gnn_outputs=gnn)
    vec.set_problem_weights(w)
    obs = vec.reset()
    assert np.array_equal(to_np(vec.new_problem_idx), fin["problem_idx0"])
    assert np.isin(fin["problem_idx0"], np.flatnonzero(w)).all()
    pre_obs = None if gnn else obs.clone()
    for t in range(T):
        if gnn and t > 0:         # the step emits the GNN input of the state the next step acts on
            assert np.array_equal(to_np(vec.out["gnn_assignment"]), tr["gs_assignment"][t]), t
            assert np.array_equal(to_np(vec.out["gnn_clause_features"]), tr["gs_clause_features"][t]), t
        elif not gnn:
            assert np.array_equal(to_np(pre_obs), tr["local_obs"][t]), t
        out = vec.step(torch.from_numpy(acts[t]).cuda())
        assert np.array_equal(to_np(out["reward"]), tr["reward"][t]), t
        assert np.array_equal(to_np(out["done"]).astype(bool), np.repeat(tr["global_done"][t][:, None],
                                                                        ref.num_agents + 1, 1)), t
        assert np.array_equal(to_np(out["solved"]).astype(bool), tr["info_solved"][t])
        assert np.array_equal(to_np(out["num_unsatisfied"]), tr["info_num_unsatisfied"][t])
        assert np.array_equal(to_np(out["episode_step"]), tr["info_episode_step"][t])
        if not gnn:
            pre_obs = out["obs"].clone()
        assert M.env.u32_to_numpy(vec.keys.act_key).tolist() == tr["act_key"][t].tolist()
    assert tr["global_done"].any()
    assert_state_equal(vec.sat_state(), fin["state"], "final ")
    if gnn:
        g = state_to_gnn_input(ref, fin["state"])
        assert np.array_equal(to_np(vec.out["gnn_assignment"]), g["assignment"])
        assert np.array_equal(to_np(vec.out["gnn_clause_features"]), g["clause_features"])
    else:
        assert np.array_equal(to_np(vec.out["obs"]), fin["obs"])
    assert np.array_equal(M.env.u32_to_numpy(vec.keys.rng), fin["rng"])
    # every auto-reset landed on a problem of positive weight
    assert np.isin(to_np(vec.sat_state().problem_idx), np.flatnonzero(w)).all()


def test_weighted_rollout_at_the_headline_shape_on_every_509th_env():
    M = _msat()
    from marl_sat_b200.synth import uniform_ksat
    n, m, B, P, T, max_steps = 100, 430, 65536, 64, 4, 2
    problems = uniform_ksat(P, n, m, 3, seed=5)
    ref = SATEnvOracle(n, m, max_steps)
    env = M.SATEnv(n, m, max_steps, verbose=False)
    q = _weights("heavy", P, 9)
    cum = np.cumsum(q.numpy())
    key0 = otf.prng_key(2024)
    vec = M.VecSATEnv(env, torch.from_numpy(problems), B, key0)
    vec.set_problem_weights(q.double())
    assert torch.equal(vec.problem_weights, q)             # quantised weights quantise to themselves
    sel = np.arange(0, B, 509)
    vec.reset()
    rng, idx0, rk0 = ocur.initial_reset_inputs(key0, B, cum)
    obs_r, st_r = ref.reset(problems[idx0[sel]], rk0[sel])
    sel_t = torch.from_numpy(sel).to(DEV)
    assert np.array_equal(to_np(vec.out["obs"][sel_t]), np.stack([obs_r[a] for a in ref.agents], 1))
    arng = np.random.default_rng(3)
    for t in range(T):
        acts = arng.integers(0, ref.max_vars_per_agent + 1, size=(B, ref.num_agents)).astype(np.int32)
        ks = ocur.rollout_keys(rng, B, cum)
        rng = ks["rng"]
        fo, st_r, rew_r, done_r, info_r = orollout.env_step_with_autoreset(
            ref, st_r, acts[sel], problems, ks["new_problem_indices"][sel], ks["reset_keys"][sel])
        out = vec.step(torch.from_numpy(acts).cuda())
        assert np.array_equal(to_np(vec.new_problem_idx), ks["new_problem_indices"])
        assert np.array_equal(to_np(out["obs"][sel_t]), fo), t
        assert np.array_equal(to_np(out["reward"][sel_t]), rew_r)
        assert np.array_equal(to_np(out["done"][sel_t]).astype(bool)[:, -1], done_r)
        for k in ("num_unsatisfied", "episode_step"):
            assert np.array_equal(to_np(out[k][sel_t]), info_r[k]), k
        assert np.array_equal(to_np(out["solved"][sel_t]).astype(bool), info_r["solved"])
        assert_state_equal(M.SATState(env, vec.bank, vec.state[sel_t].contiguous(), True), st_r, f"step {t} ")


# ---------------------------------------------------------------------------------------------- weights off / one-hot
def _run(vec, actions):
    rows = []
    for a in actions:
        out = vec.step(a)
        rows.append({k: out[k].clone() for k in ("obs", "reward", "done", "solved", "num_unsatisfied", "episode_step")
                     if out.get(k) is not None})
    return rows


def test_weights_none_is_bit_identical_to_never_weighted():
    M = _msat()
    from marl_sat_b200.synth import uniform_ksat
    n, m, B, P, max_steps = 50, 218, 300, 9, 3
    env = M.SATEnv(n, m, max_steps, verbose=False)
    bank = env.make_bank(uniform_ksat(P, n, m, 3, seed=4))
    g = torch.Generator(device="cuda").manual_seed(2)
    actions = [torch.randint(0, 8, (B, env.num_agents), generator=g, device="cuda", dtype=torch.int32) for _ in range(8)]
    plain = M.VecSATEnv(env, bank, B, otf.prng_key(9))
    toggled = M.VecSATEnv(env, bank, B, otf.prng_key(9))
    toggled.set_problem_weights(np.arange(P, dtype=np.float64))
    toggled.set_problem_weights(None)
    assert toggled.problem_weights is None
    plain.reset()
    toggled.reset()
    assert torch.equal(plain.state, toggled.state) and torch.equal(plain.out["obs"], toggled.out["obs"])
    for t, (a, b) in enumerate(zip(_run(plain, actions), _run(toggled, actions))):
        for k in a:
            assert torch.equal(a[k], b[k]), (t, k)
    assert torch.equal(plain.state, toggled.state) and torch.equal(plain.keys.chain, toggled.keys.chain)
    assert getattr(toggled, "_fast_args", None) is not None          # the fused one-launch step ran


def test_one_hot_weights_put_every_reset_on_that_problem():
    M = _msat()
    from marl_sat_b200.synth import uniform_ksat
    n, m, B, P, q, max_steps = 20, 91, 500, 12, 7, 2
    env = M.SATEnv(n, m, max_steps, verbose=False)
    bank = env.make_bank(uniform_ksat(P, n, m, 3, seed=1))
    vec = M.VecSATEnv(env, bank, B, otf.prng_key(4))
    vec.set_problem_weights(np.eye(P)[q])
    vec.reset()
    assert bool((vec.sat_state().problem_idx == q).all())
    vec.set_problem_weights(None)
    g = torch.Generator(device="cuda").manual_seed(0)
    for _ in range(3):                                  # uniform auto-resets spread the batch over the bank again
        vec.step(torch.randint(0, 6, (B, env.num_agents), generator=g, device="cuda", dtype=torch.int32))
    assert len(torch.unique(vec.sat_state().problem_idx)) > 1
    vec.set_problem_weights(np.eye(P)[q])
    resets = 0
    for _ in range(2 * max_steps + 1):
        out = vec.step(torch.randint(0, 6, (B, env.num_agents), generator=g, device="cuda", dtype=torch.int32))
        done = out["done"][:, -1].bool()
        resets += int(done.sum())
        assert bool((vec.sat_state().problem_idx[done] == q).all())
    assert resets >= B and bool((vec.sat_state().problem_idx == q).all())


# ---------------------------------------------------------------------------------------------- statistics
@pytest.mark.parametrize("P", [1, 7, 800, 1024, 1025, 65536])
def test_stats_match_the_oracle_on_random_rollouts(P):
    M = _msat()
    rng = np.random.default_rng(P)
    T, B = 37, 1000
    done = rng.random((T, B)) < 0.3
    solved = rng.random((T, B)) < 0.5
    nu = rng.integers(-2 ** 31, 2 ** 31, (T, B)).astype(np.int32)        # the sums stay exact for any int32
    es = rng.integers(-2 ** 31, 2 ** 31, (T, B)).astype(np.int32)
    nu[:, ::3] = rng.integers(0, 400, (T, (B + 2) // 3))
    pidx = rng.integers(-5, P + 5, (T, B)).astype(np.int32)
    pidx[:, :200] = rng.integers(0, min(P, 3), (T, 200))                  # hot problems inside a warp
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(DEV)
    got = M.problem_stats(t(pidx), t(done), t(solved.astype(np.uint8)), t(nu), t(es), P)
    exp = ocur.problem_stats(pidx, done, solved, nu, es, P)
    assert got.dtype == torch.int64 and np.array_equal(to_np(got), exp)
    # two calls accumulate
    again = M.problem_stats(t(pidx), t(done), t(solved), t(nu), t(es), P, stats=got)
    assert again is got and np.array_equal(to_np(got), 2 * exp)


def test_stats_contention_one_problem_every_row_done():
    M = _msat()
    T, B = 512, 4096
    ones = torch.ones((T, B), dtype=torch.uint8, device=DEV)
    steps = torch.arange(T * B, dtype=torch.int32, device=DEV).reshape(T, B) % 97
    got = M.problem_stats(torch.zeros((T, B), dtype=torch.int32, device=DEV), ones, ones,
                          torch.full((T, B), 3, dtype=torch.int32, device=DEV), steps, 1)
    assert got.tolist() == [[T * B, T * B, 3 * T * B, int(steps.sum())]]


def test_buffer_stats_equal_dense_indices_and_rollout_metrics():
    M = _msat()
    from marl_sat_b200.synth import uniform_ksat
    n, m, B, P, T, max_steps = 20, 91, 777, 23, 16, 4
    env = M.SATEnv(n, m, max_steps, verbose=False)
    bank = env.make_bank(uniform_ksat(P, n, m, 3, seed=3))
    vec = M.VecSATEnv(env, bank, B, otf.prng_key(8), compact_outputs=True)
    vec.set_problem_weights(np.linspace(0.0, 1.0, P))
    vec.reset()
    buf = M.RolloutBuffer(env, bank, T, B)
    g = torch.Generator(device="cuda").manual_seed(1)
    actions = torch.randint(0, 6, (T, B, env.num_agents), generator=g, device="cuda", dtype=torch.int32)
    buf.collect(vec, lambda t, v: (actions[t], None, None))
    stats = buf.problem_stats()
    dense = torch.stack([buf.pre_step_state(t).problem_idx for t in range(T)]).contiguous()
    assert torch.equal(stats, M.problem_stats(dense, buf.global_done, buf.solved, buf.num_unsatisfied,
                                              buf.episode_step, P))
    sums = M.rollout_metric_sums(buf.reward, buf.global_done, buf.solved, buf.num_unsatisfied, buf.episode_step)
    assert to_np(stats.sum(0)).tolist() == [int(x) for x in to_np(sums[1:5])]
    assert int(stats[0, 0]) == 0 and int(stats[:, 0].sum()) > 0       # problem 0 has weight 0
    total = torch.zeros((P, 4), dtype=torch.int64, device=DEV)
    buf.problem_stats(total)
    buf.problem_stats(total)
    assert torch.equal(total, 2 * stats)


# ---------------------------------------------------------------------------------------------- graph / checkpoint / refusals
def test_graph_captured_weighted_step_replays_to_the_eager_result():
    M = _msat()
    from marl_sat_b200.synth import uniform_ksat
    n, m, B, P, G = 50, 218, 1000, 16, 4
    env = M.SATEnv(n, m, 3, verbose=False)
    bank = env.make_bank(uniform_ksat(P, n, m, 3, seed=7))
    acts = torch.randint(0, 8, (G, B, env.num_agents), device=DEV, dtype=torch.int32)
    w1, w2 = np.arange(P, dtype=np.float64), np.eye(P)[5] + np.eye(P)[11] * 3
    graphed = M.VecSATEnv(env, bank, B, otf.prng_key(1))
    graphed.set_problem_weights(w1)
    graphed.reset()
    state0, chain0, cur0 = graphed.state.clone(), graphed.keys._bufs.clone(), graphed.keys._cur
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                       # warm-up outside the capture
        for t in range(G):
            graphed.step(acts[t])
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for t in range(G):
            graphed.step(acts[t])
    assert graphed.keys._cur == cur0                    # an even number of steps: the chain buffers line up again
    for w in (w1, w2):
        graphed.set_problem_weights(w)                  # in place: no re-capture
        graphed.state.copy_(state0)
        graphed.keys._bufs.copy_(chain0)
        graph.replay()
        eager = M.VecSATEnv(env, bank, B, otf.prng_key(1))
        eager.set_problem_weights(w)
        eager.state.copy_(state0)
        eager.keys._bufs.copy_(chain0)
        eager.keys._cur = cur0
        for t in range(G):
            eager.step(acts[t])
        torch.cuda.synchronize()
        assert torch.equal(graphed.state, eager.state) and torch.equal(graphed.out["obs"], eager.out["obs"])
        assert torch.equal(graphed.out["_block"], eager.out["_block"])
    assert bool(torch.isin(graphed.sat_state().problem_idx, torch.tensor([5, 11], device=DEV)).any())


def test_checkpoint_with_weights_round_trips():
    M = _msat()
    from marl_sat_b200.synth import uniform_ksat
    n, m, B, P, max_steps, t = 20, 91, 50, 7, 3, 5
    env = M.SATEnv(n, m, max_steps, verbose=False)
    bank = env.make_bank(uniform_ksat(P, n, m, 3, seed=31))
    w = np.array([0.0, 1.0, 0.0, 4.0, 0.5, 0.0, 2.0])
    g = torch.Generator(device="cuda").manual_seed(1)
    actions = [torch.randint(0, 5, (B, env.num_agents), generator=g, device="cuda", dtype=torch.int32)
               for _ in range(2 * t)]
    full = M.VecSATEnv(env, bank, B, otf.prng_key(77))
    full.set_problem_weights(w)
    full.reset()
    ref_rows = _run(full, actions)

    plain = M.VecSATEnv(env, bank, B, otf.prng_key(77))
    plain.reset()
    assert "problem_weights" not in plain.state_dict()         # unweighted checkpoints keep their keys
    shards = [M.VecSATEnv(env, bank, B, otf.prng_key(77), world_size=2, rank=r) for r in range(2)]
    for s in shards:
        s.set_problem_weights(w)
        s.reset()
    for a in actions[:t]:
        for s in shards:
            s.step(a[s.env_offset:s.env_offset + s.num_envs].contiguous())
    sds = [s.state_dict() for s in shards]
    assert torch.equal(sds[0]["problem_weights"], M.problem_weights(w))
    merged = M.merge_state_dicts(sds)
    assert torch.equal(merged["problem_weights"], M.problem_weights(w))
    single = M.VecSATEnv(env, bank, B, otf.prng_key(0))
    single.load_state_dict(merged)
    assert torch.equal(single.problem_weights, M.problem_weights(w))
    rows = _run(single, actions[t:])
    for i, (a, b) in enumerate(zip(rows, ref_rows[t:])):
        for k in a:
            assert torch.equal(a[k], b[k]), (i, k)
    assert torch.equal(single.state, full.state)
    # a checkpoint without weights restores the uniform draw; shards with different weights do not merge
    single.load_state_dict(plain.state_dict())
    assert single.problem_weights is None
    other = dict(sds[1], problem_weights=M.problem_weights(w[::-1].copy()))
    with pytest.raises(ValueError, match="weights"):
        M.merge_state_dicts([sds[0], other])
    with pytest.raises(ValueError, match="weights"):
        M.merge_state_dicts([sds[0], {k: v for k, v in sds[1].items() if k != "problem_weights"}])


def test_fused_multi_step_and_host_paths_refuse_weights():
    M = _msat()
    from marl_sat_b200.synth import uniform_ksat
    env = M.SATEnv(20, 91, 4, verbose=False)
    vec = M.VecSATEnv(env, env.make_bank(uniform_ksat(5, 20, 91, 3, seed=2)), 64, otf.prng_key(3))
    vec.set_problem_weights([1.0, 0.0, 1.0, 0.0, 1.0])
    vec.reset()
    acts = torch.zeros((2, 64, env.num_agents), dtype=torch.int32, device=DEV)
    with pytest.raises(ValueError, match="weights"):
        vec.steps(acts, vec.alloc_multi_step_outputs(2))
    with pytest.raises(ValueError, match="weights"):
        vec.step_host(vec.alloc_host_io())
    slots = vec.alloc_async_io(1)
    with pytest.raises(ValueError, match="weights"):
        vec.step_host_async(0, slots[0])
    vec.close()
    with pytest.raises(ValueError):
        vec.set_problem_weights([1.0, 2.0])                      # wrong length for this bank


# ---------------------------------------------------------------------------------------------- two ranks
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _stats_setup(M, world, rank):
    from marl_sat_b200.synth import uniform_ksat
    n, m, Bg, P, T = 20, 40, 48, 7, 12
    env = M.SATEnv(n, m, 4, verbose=False)
    bank = env.make_bank(uniform_ksat(P, n, m, 3, seed=3))
    vec = M.VecSATEnv(env, bank, Bg, M.prng_key(11), world_size=world, rank=rank, compact_outputs=True)
    vec.set_problem_weights([1.0, 2.0, 0.0, 1.0, 3.0, 0.5, 1.0])
    vec.reset()
    g = torch.Generator(device="cuda").manual_seed(5)
    actions = torch.randint(0, 5, (T, Bg, env.num_agents), generator=g, device="cuda", dtype=torch.int32)
    buf = M.RolloutBuffer(env, bank, T, vec.num_envs)
    sl = slice(vec.env_offset, vec.env_offset + vec.num_envs)
    buf.collect(vec, lambda t, v: (actions[t, sl], None, None))
    return buf


def _stats_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import marl_sat_b200 as M
        buf = _stats_setup(M, world, rank)
        local = buf.problem_stats()
        total = torch.zeros_like(local)
        buf.problem_stats(total)
        buf.problem_stats(total)                       # running totals are not all-reduced again
        out = [None] * world
        dist.all_gather_object(out, (local.cpu().numpy(), total.cpu().numpy()))
        if rank == 0:
            q.put(out)
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_two_ranks_all_reduce_the_stats_of_the_full_batch():
    import torch.multiprocessing as mp
    M = _msat()
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.SimpleQueue()
    port = _free_port()
    procs = [ctx.Process(target=_stats_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    gathered = q.get()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    full = to_np(_stats_setup(M, 1, 0).problem_stats())
    assert full[:, 0].sum() > 0 and full[2, 0] == 0
    for local, total in gathered:
        assert np.array_equal(local, full)
        assert np.array_equal(total, 2 * full)
