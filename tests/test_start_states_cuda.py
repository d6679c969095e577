"""GPU tests of the start states (``msat_apply_start_states``, ``VecSATEnv.set_start_states``): rollouts with starts
against the NumPy oracle (``oracle/start_states.py``) bit for bit, WalkSAT
solutions as exact starts, no change where starts are unused, sharding, checkpoints, graph capture and refusals."""
import numpy as np
import pytest
import torch

from oracle import start_states as ostart
from oracle import rollout as orollout
from oracle import threefry as otf
from oracle.sat_env import SATEnvOracle
from tests.util import assert_state_equal, to_np

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")


def _msat():
    import marl_sat_b200 as M
    return M


def _formulas(kind, P, n, m, k, seed):
    from marl_sat_b200.synth import mixed_ksat, uniform_ksat
    return uniform_ksat(P, n, m, k, seed) if kind == "uniform" else mixed_ksat(P, n, m, 3, k, seed)


def _actions(rng, ref, T, B):
    if ref.action_mode == 0:
        return rng.integers(0, ref.max_vars_per_agent + 2, size=(T, B, ref.num_agents)).astype(np.int32)
    return rng.integers(0, 2, size=(T, B, ref.num_agents, ref.max_vars_per_agent)).astype(np.int32)


def _starts(P, n, seed):
    """Random start assignments, q cycling over {0, 0.05, 0.5}, and every other problem without a start."""
    rng = np.random.default_rng(seed)
    start = rng.integers(0, 2, (P, n)).astype(np.int32)
    q = np.array([0.0, 0.05, 0.5])[np.arange(P) % 3]
    has = (np.arange(P) % 2 == 0).astype(np.uint8)
    return start, q, has


# ---------------------------------------------------------------------------------------------- oracle parity
# (name, n, m, k, vars_per_agent, kind, action_mode)
SHAPES = [("uf20-91 mode 0", 20, 91, 3, None, "uniform", 0), ("uf20-91 mode 1", 20, 91, 3, None, "uniform", 1),
          ("uf50-218 uneven", 50, 218, 3, None, "uniform", 0), ("mixed k3-7 vpa7", 40, 170, 7, 7, "mixed", 0),
          ("uf100-430", 100, 430, 3, None, "uniform", 0)]


@pytest.mark.parametrize("outputs", ["int32", "int8", "gnn"])
@pytest.mark.parametrize("clause_update", ["full", "incremental"])
@pytest.mark.parametrize("name,n,m,k,vpa,kind,mode", SHAPES, ids=[s[0] for s in SHAPES])
def test_rollout_with_starts_matches_the_oracle(name, n, m, k, vpa, kind, mode, clause_update, outputs):
    M = _msat()
    B, P, T, max_steps = 96, 12, 9, 3
    problems = _formulas(kind, P, n, m, k, seed=n + k)
    ref = SATEnvOracle(n, m, max_steps, vars_per_agent=vpa, action_mode=mode)
    env = M.SATEnv(n, m, max_steps, vars_per_agent=vpa, action_mode=mode, verbose=False, clause_update=clause_update,
                   obs_dtype="int8" if outputs == "int8" else "int32")
    start, q, has = _starts(P, n, seed=n)
    thr = ostart.quantize_flip_prob(q)
    key0 = otf.prng_key(7 + mode)
    acts = _actions(np.random.default_rng(mode + n), ref, T, B)
    tr, fin = ostart.rollout_T(ref, problems, key0, acts, (start, thr, has))
    gnn = outputs == "gnn"
    vec = M.VecSATEnv(env, torch.from_numpy(problems), B, key0, emit_obs=not gnn, gnn_outputs=gnn)
    vec.set_start_states(start, q, has_start=has)
    assert vec.start_states.flip_thr.tolist() == thr.tolist()
    obs = vec.reset()
    if not gnn:
        assert np.array_equal(to_np(obs).astype(np.int32), tr["local_obs"][0])
    for t in range(T):
        if gnn and t > 0:
            assert np.array_equal(to_np(vec.out["gnn_assignment"]), tr["gs_assignment"][t]), t
            assert np.array_equal(to_np(vec.out["gnn_clause_features"]), tr["gs_clause_features"][t]), t
        out = vec.step(torch.from_numpy(acts[t]).cuda())
        assert np.array_equal(to_np(out["reward"])[:, 0], tr["reward"][t][:, 0]), t
        assert np.array_equal(to_np(out["done"])[:, -1].astype(bool), tr["global_done"][t]), t
        assert np.array_equal(to_np(out["solved"]).astype(bool), tr["info_solved"][t])
        assert np.array_equal(to_np(out["num_unsatisfied"]), tr["info_num_unsatisfied"][t])
        assert np.array_equal(to_np(out["episode_step"]), tr["info_episode_step"][t])
        st = vec.sat_state()
        if t + 1 < T:
            assert np.array_equal(to_np(st.variable_assignments), tr["gs_assignment"][t + 1]), t
            if not gnn:
                assert np.array_equal(to_np(out["obs"]).astype(np.int32), tr["local_obs"][t + 1]), t
        # the policy input the step left equals what get_obs / gnn_dynamic make of the state
        if gnn:
            a, cf = M.dynamic_features(st)
            assert torch.equal(a, vec.out["gnn_assignment"]) and torch.equal(cf, vec.out["gnn_clause_features"])
        else:
            assert torch.equal(env.get_obs_array(st), out["obs"])
    assert tr["global_done"].any()
    assert_state_equal(vec.sat_state(), fin["state"], "final ")
    # restarted envs on problems with a start sit at start XOR flips; q = 0 problems exactly at the start
    st = vec.sat_state()
    fresh = to_np(st.step) == 0
    p = to_np(st.problem_idx)
    exact = fresh & (has[p] != 0) & (q[p] == 0.0)
    if exact.any():
        assert np.array_equal(to_np(st.variable_assignments)[exact], start[p[exact]])


def test_headline_shape_on_every_509th_env():
    M = _msat()
    n, m, B, P, T, max_steps = 100, 430, 65536, 64, 4, 2
    problems = _formulas("uniform", P, n, m, 3, seed=5)
    ref = SATEnvOracle(n, m, max_steps)
    env = M.SATEnv(n, m, max_steps, verbose=False)
    start, q, has = _starts(P, n, seed=1)
    thr = ostart.quantize_flip_prob(q)
    key0 = otf.prng_key(2024)
    vec = M.VecSATEnv(env, torch.from_numpy(problems), B, key0)
    vec.set_start_states(start, q, has_start=has)
    sel = np.arange(0, B, 509)
    sel_t = torch.from_numpy(sel).to(DEV)
    vec.reset()
    rng, idx0, rk0 = orollout.initial_reset_inputs(key0, B, P)
    obs_r, st_r = ref.reset(problems[idx0[sel]], rk0[sel])
    obs_r = np.stack([obs_r[a] for a in ref.agents], 1)
    pidx = idx0[sel].astype(np.int64)
    st_r, obs_r = ostart.apply_start_states(ref, st_r, obs_r, pidx, rk0[sel], (start, thr, has))
    assert np.array_equal(to_np(vec.out["obs"][sel_t]), obs_r)
    arng = np.random.default_rng(3)
    for t in range(T):
        acts = arng.integers(0, ref.max_vars_per_agent + 1, size=(B, ref.num_agents)).astype(np.int32)
        ks = orollout.rollout_keys(rng, B, P)
        rng = ks["rng"]
        fo, st_r, rew_r, done_r, info_r = orollout.env_step_with_autoreset(
            ref, st_r, acts[sel], problems, ks["new_problem_indices"][sel], ks["reset_keys"][sel])
        pidx = np.where(done_r, ks["new_problem_indices"][sel], pidx)
        st_r, fo = ostart.apply_start_states(ref, st_r, fo, pidx, ks["reset_keys"][sel], (start, thr, has))
        out = vec.step(torch.from_numpy(acts).cuda())
        assert np.array_equal(to_np(out["obs"][sel_t]), fo), t
        assert np.array_equal(to_np(out["reward"][sel_t]), rew_r)
        assert np.array_equal(to_np(out["num_unsatisfied"][sel_t]), info_r["num_unsatisfied"])
        assert_state_equal(M.SATState(env, vec.bank, vec.state[sel_t].contiguous(), True), st_r, f"step {t} ")


# ---------------------------------------------------------------------------------------------- WalkSAT starts
def test_q0_starts_from_walksat_solutions_land_on_solutions():
    M = _msat()
    n, m, P, B, max_steps = 20, 91, 32, 512, 4
    env = M.SATEnv(n, m, max_steps, verbose=False)
    bank = env.make_bank(_formulas("uniform", P, n, m, 3, seed=11))
    idx = torch.arange(P, dtype=torch.int32, device=DEV)
    keys = M.env.as_u32_tensor(otf.split(otf.prng_key(5), P), DEV)
    _, st = env.reset_from_bank(bank, idx, keys, want_obs=False)
    res = M.walksat(st, keys, 10_000)
    solved = res.solved.cpu()
    assert int(solved.sum()) >= P // 2
    vec = M.VecSATEnv(env, bank, B, otf.prng_key(6))
    vec.set_problem_weights(solved.double())
    vec.set_start_states(res.state.variable_assignments, 0.0, has_start=solved)
    vec.reset()
    assert bool((vec.sat_state().num_unsatisfied == 0).all())
    g = torch.Generator(device="cuda").manual_seed(0)
    restarts = 0
    for _ in range(3 * max_steps):
        out = vec.step(torch.randint(0, env.max_vars_per_agent + 1, (B, env.num_agents), generator=g, device=DEV,
                                     dtype=torch.int32))
        done = out["done"][:, -1].bool()
        restarts += int(done.sum())
        st = vec.sat_state()
        assert bool((st.num_unsatisfied[done] == 0).all()) and bool((st.step[done] == 0).all())
    assert restarts >= B


# ---------------------------------------------------------------------------------------------- unused starts
def _run(vec, actions):
    rows = []
    for a in actions:
        out = vec.step(a)
        rows.append({k: out[k].clone() for k in ("obs", "reward", "done", "solved", "num_unsatisfied", "episode_step")
                     if out.get(k) is not None})
    return rows


def _setup(seed=4, n=50, m=218, P=9, max_steps=3):
    M = _msat()
    env = M.SATEnv(n, m, max_steps, verbose=False)
    bank = env.make_bank(_formulas("uniform", P, n, m, 3, seed=seed))
    return M, env, bank


def test_unused_starts_are_bit_identical_to_never_setting_them():
    M, env, bank = _setup()
    B, P, n = 300, 9, 50
    g = torch.Generator(device="cuda").manual_seed(2)
    actions = [torch.randint(0, 8, (B, env.num_agents), generator=g, device=DEV, dtype=torch.int32) for _ in range(8)]
    plain = M.VecSATEnv(env, bank, B, otf.prng_key(9))
    toggled = M.VecSATEnv(env, bank, B, otf.prng_key(9))
    toggled.set_start_states(np.ones((P, n), np.int32), 0.1)
    toggled.set_start_states(None)
    assert toggled.start_states is None
    never = M.VecSATEnv(env, bank, B, otf.prng_key(9))             # set, but on no problem
    never.set_start_states(np.ones((P, n), np.int32), 0.1, has_start=np.zeros(P, np.uint8))
    for v in (plain, toggled, never):
        v.reset()
    assert torch.equal(plain.state, toggled.state) and torch.equal(plain.state, never.state)
    assert torch.equal(plain.out["obs"], never.out["obs"])
    ref = _run(plain, actions)
    for other in (toggled, never):
        for t, (a, b) in enumerate(zip(ref, _run(other, actions))):
            for k in a:
                assert torch.equal(a[k], b[k]), (t, k)
        assert torch.equal(plain.state, other.state) and torch.equal(plain.keys.chain, other.keys.chain)


# ---------------------------------------------------------------------------------------------- sharding / resume
def _sharded_run(M, env, bank, Bg, world, starts, actions, key=otf.prng_key(21)):
    shards = [M.VecSATEnv(env, bank, Bg, key, world_size=world, rank=r) for r in range(world)]
    for s in shards:
        s.set_start_states(*starts)
        s.reset()
    rows = []
    for a in actions:
        outs = [s.step(a[s.env_offset:s.env_offset + s.num_envs].contiguous()) for s in shards]
        rows.append({k: torch.cat([o[k] for o in outs]) for k in ("obs", "reward", "done", "num_unsatisfied")})
    return shards, rows


def test_sharded_runs_equal_the_single_device_run():
    M, env, bank = _setup(n=20, m=91, P=10, max_steps=2)
    Bg = 301
    start, q, has = _starts(10, 20, seed=3)
    g = torch.Generator(device="cuda").manual_seed(4)
    actions = [torch.randint(0, 7, (Bg, env.num_agents), generator=g, device=DEV, dtype=torch.int32) for _ in range(7)]
    one, ref = _sharded_run(M, env, bank, Bg, 1, (start, q, has), actions)
    for world in (2, 3):
        shards, rows = _sharded_run(M, env, bank, Bg, world, (start, q, has), actions)
        for t, (a, b) in enumerate(zip(ref, rows)):
            for k in a:
                assert torch.equal(a[k], b[k]), (world, t, k)
        assert torch.equal(torch.cat([s.state for s in shards]), one[0].state)


def test_checkpoint_with_starts_resumes_exactly_into_one_and_three_shards():
    M, env, bank = _setup(n=20, m=91, P=7, max_steps=3)
    B, t = 50, 5
    start, q, has = _starts(7, 20, seed=8)
    g = torch.Generator(device="cuda").manual_seed(1)
    actions = [torch.randint(0, 5, (B, env.num_agents), generator=g, device=DEV, dtype=torch.int32) for _ in range(2 * t)]
    full = M.VecSATEnv(env, bank, B, otf.prng_key(77))
    full.set_start_states(start, q, has_start=has)
    full.reset()
    ref_rows = _run(full, actions)

    half = M.VecSATEnv(env, bank, B, otf.prng_key(77))
    half.set_start_states(start, q, has_start=has)
    half.reset()
    _run(half, actions[:t])
    sd = half.state_dict()
    assert set(sd["start_states"]) == {"words", "flip_thr", "has_start"}
    for world in (1, 3):
        shards = [M.VecSATEnv(env, bank, B, otf.prng_key(0), world_size=world, rank=r) for r in range(world)]
        for s in shards:
            s.load_state_dict(sd)
            assert s.start_states.flip_thr.tolist() == ostart.quantize_flip_prob(q).tolist()
        for i, a in enumerate(actions[t:]):
            outs = [s.step(a[s.env_offset:s.env_offset + s.num_envs].contiguous()) for s in shards]
            for k in ("obs", "reward", "done", "num_unsatisfied", "episode_step"):
                assert torch.equal(torch.cat([o[k] for o in outs]), ref_rows[t + i][k]), (world, i, k)
        assert torch.equal(torch.cat([s.state for s in shards]), full.state)
        if world == 3:
            merged = M.merge_state_dicts([s.state_dict() for s in shards])
            assert all(torch.equal(merged["start_states"][k], sd["start_states"][k]) for k in sd["start_states"])
            other = dict(shards[1].state_dict())
            other["start_states"] = dict(other["start_states"], has_start=1 - other["start_states"]["has_start"])
            with pytest.raises(ValueError, match="start states"):
                M.merge_state_dicts([shards[0].state_dict(), other, shards[2].state_dict()])
    # a checkpoint without starts clears them
    plain = M.VecSATEnv(env, bank, B, otf.prng_key(77))
    plain.reset()
    assert "start_states" not in plain.state_dict()
    half.load_state_dict(plain.state_dict())
    assert half.start_states is None


# ---------------------------------------------------------------------------------------------- graph / refusals
def test_graph_captured_step_picks_up_a_new_q_without_recapture():
    M, env, bank = _setup(n=50, m=218, P=16, max_steps=2)
    B, G, P, n = 1000, 4, 16, 50
    acts = torch.randint(0, 8, (G, B, env.num_agents), device=DEV, dtype=torch.int32)
    start = np.random.default_rng(0).integers(0, 2, (P, n)).astype(np.int32)
    graphed = M.VecSATEnv(env, bank, B, otf.prng_key(1))
    graphed.set_start_states(start, 0.3)
    graphed.reset()
    state0, chain0, cur0 = graphed.state.clone(), graphed.keys._bufs.clone(), graphed.keys._cur
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for t in range(G):
            graphed.step(acts[t])
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for t in range(G):
            graphed.step(acts[t])
    for q in (0.0, 0.02, np.linspace(0.0, 1.0, P)):
        graphed.set_start_states(start, q)                           # in place: no re-capture
        graphed.state.copy_(state0)
        graphed.keys._bufs.copy_(chain0)
        graph.replay()
        eager = M.VecSATEnv(env, bank, B, otf.prng_key(1))
        eager.set_start_states(start, q)
        eager.state.copy_(state0)
        eager.keys._bufs.copy_(chain0)
        eager.keys._cur = cur0
        for t in range(G):
            eager.step(acts[t])
        torch.cuda.synchronize()
        assert torch.equal(graphed.state, eager.state) and torch.equal(graphed.out["obs"], eager.out["obs"])
        st = eager.sat_state()
        if np.isscalar(q) and q == 0.0:
            fresh = to_np(st.step) == 0
            assert fresh.any()
            assert np.array_equal(to_np(st.variable_assignments)[fresh], start[to_np(st.problem_idx)[fresh]])


def test_fused_multi_step_and_host_paths_refuse_starts():
    M, env, bank = _setup(n=20, m=91, P=5, max_steps=4)
    vec = M.VecSATEnv(env, bank, 64, otf.prng_key(3))
    vec.set_start_states(np.zeros((5, 20), np.int32), 0.1)
    vec.reset()
    acts = torch.zeros((2, 64, env.num_agents), dtype=torch.int32, device=DEV)
    with pytest.raises(ValueError, match="start states"):
        vec.steps(acts, vec.alloc_multi_step_outputs(2))
    with pytest.raises(ValueError, match="start states"):
        vec.step_host(vec.alloc_host_io())
    slots = vec.alloc_async_io(1)
    with pytest.raises(ValueError, match="start states"):
        vec.step_host_async(0, slots[0])
    vec.close()
    with pytest.raises(ValueError, match="start assignments"):
        vec.set_start_states(np.zeros((4, 20), np.int32))            # wrong row count for this bank


def test_apply_start_states_writes_obs_and_gnn_outputs_of_one_call():
    """Observations and GNN inputs in one call (two launches): both equal get_obs / gnn_dynamic of the new state,
    and rows of envs that did not restart are untouched."""
    M, env, bank = _setup(n=20, m=91, P=6, max_steps=5)
    B, P, n = 200, 6, 20
    vec = M.VecSATEnv(env, bank, B, otf.prng_key(12))
    vec.reset()
    vec.step(torch.zeros((B, env.num_agents), dtype=torch.int32, device=DEV))
    steps = torch.arange(B, device=DEV, dtype=torch.int32) % 2                 # half the envs "just restarted"
    vec.set_episode_steps(steps)
    table = M.curriculum.start_table(np.ones((P, n), np.int32), 0.05, has_start=np.arange(P) % 3 != 0)
    dev = {k: v.to(DEV) for k, v in zip(("words", "thr", "has"), (table.words, table.flip_thr.to(torch.int32),
                                                                  table.has_start))}
    obs = torch.full_like(vec.out["obs"], 7)
    ga = torch.full((B, n), 7, dtype=torch.int32, device=DEV)
    cf = torch.full((B, 91, 3), 7.0, device=DEV)
    before = vec.state.clone()
    rk = M.env.as_u32_tensor(otf.prng_key(99), DEV)
    M._lib.check(env._lib.msat_apply_start_states(
        bank.plan.handle, bank.data.data_ptr(), P, vec.state.data_ptr(), rk.data_ptr(), B, 0, dev["words"].data_ptr(),
        dev["thr"].data_ptr(), dev["has"].data_ptr(), obs.data_ptr(), ga.data_ptr(), cf.data_ptr(), B,
        torch.cuda.current_stream().cuda_stream), "msat_apply_start_states")
    st = vec.sat_state()
    p = to_np(st.problem_idx)
    sel = (to_np(steps) == 0) & (p % 3 != 0)
    assert sel.any() and (~sel).any()
    assert torch.equal(vec.state[torch.from_numpy(~sel).to(DEV)], before[torch.from_numpy(~sel).to(DEV)])
    s = torch.from_numpy(sel).to(DEV)
    a, f = M.dynamic_features(st)
    assert torch.equal(obs[s], env.get_obs_array(st)[s]) and bool((obs[~s] == 7).all())
    assert torch.equal(ga[s], a[s]) and bool((ga[~s] == 7).all())
    assert torch.equal(cf[s], f[s]) and bool((cf[~s] == 7.0).all())
    keys = otf.split(otf.prng_key(99), B)
    exp = ostart.start_assignments(np.ones((P, n), np.int32), to_np(table.flip_thr), p[sel], keys[sel])
    assert np.array_equal(to_np(st.variable_assignments)[sel], exp)
