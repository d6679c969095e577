"""GPU tests of the state import (``msat_import_state``, ``SATEnv.import_state``) and of resumable, reshardable
rollout checkpoints (``VecSATEnv.state_dict`` / ``load_state_dict``).

* parity: an imported state equals the oracle state built from the same (clauses, assignment, step, done) in all
  nine ``SATState`` leaves and in the observations, and keeps matching the oracle over further steps;
* exact inverse: reset / rollout -> export -> import reproduces every packed word (padding included) and the
  observations, for every group size, both observation dtypes and both clause-update modes;
* resume / reshard: a rollout interrupted by a checkpoint continues with exactly the outputs of the uninterrupted
  run, also on 2 or 3 shards and on a plan with the other clause-update mode.
"""
import numpy as np
import pytest
import torch

from oracle import threefry as otf
from oracle.sat_env import SATEnvOracle, SATState as OracleState, _jax_gather_index
from tests.test_parity_cuda import SHAPES
from tests.util import assert_obs_equal, assert_state_equal, to_np

pytestmark = pytest.mark.gpu


def _msat():
    import marl_sat_b200 as M
    return M


def _formulas(kind, P, n, m, k, seed):
    from marl_sat_b200.synth import mixed_ksat, uniform_ksat
    if kind == "uniform":
        return uniform_ksat(P, n, m, k, seed)
    return mixed_ksat(P, n, m, 3 if kind == "mixed" else 2, k, seed)


def _keys(B, seed):
    return np.random.default_rng(seed).integers(0, 2 ** 32, size=(B, 2), dtype=np.uint64).astype(np.uint32)


def _actions(rng, ref, B):
    if ref.action_mode == 0:
        return rng.integers(0, ref.max_vars_per_agent + 2, size=(B, ref.num_agents)).astype(np.int32)
    return rng.integers(0, 2, size=(B, ref.num_agents, ref.max_vars_per_agent)).astype(np.int32)


def oracle_import(ref: SATEnvOracle, clauses, assign, step, done) -> OracleState:
    """The reference ``SATState`` (env:13-24) of (clauses, assignment, step, done): observation maps and
    satisfaction recomputed exactly as ``reset`` does (env:158-181), step and done as given."""
    clauses = np.asarray(clauses, np.int32)
    assign = (np.asarray(assign) != 0).astype(np.int32)
    acm, anm = ref.compute_observation_maps(clauses)
    status, num_unsat = ref.calculate_satisfaction(assign, clauses)
    l2a = ref.variable_to_agent_idx[_jax_gather_index(np.abs(clauses) - 1, ref.num_vars)]
    return OracleState(variable_assignments=assign, clauses_satisfied_status=status, num_unsatisfied=num_unsat,
                       step=np.asarray(step, np.int32), done=np.repeat(np.asarray(done, bool)[:, None], ref.num_agents, 1),
                       clauses=clauses, agent_clause_masks=acm, agent_neighbor_masks=anm,
                       literal_to_agent_idx=l2a.astype(np.int32), action_mask=ref.action_mask)


# ---------------------------------------------------------------------------------------------- oracle parity
@pytest.mark.parametrize("name,n,m,k,vpa,kind", SHAPES, ids=[s[0] for s in SHAPES])
@pytest.mark.parametrize("mode", [0, 1])
def test_import_matches_oracle_and_keeps_stepping(name, n, m, k, vpa, kind, mode):
    M = _msat()
    B, max_steps = (37 if n < 200 else 11), 4
    clauses = _formulas(kind, B, n, m, k, seed=n * 13 + m)
    rng = np.random.default_rng(n + m + 17 * mode)
    assign = rng.integers(0, 2, size=(B, n)).astype(np.int32)
    step = rng.integers(0, max_steps + 4, size=B).astype(np.int32)          # [0, max_steps + 3]
    done = rng.random(B) < 0.4
    ref = SATEnvOracle(n, m, max_steps, vars_per_agent=vpa, action_mode=mode)
    env = M.SATEnv(n, m, max_steps, vars_per_agent=vpa, action_mode=mode, verbose=False)
    st_r = oracle_import(ref, clauses, assign, step, done)
    bank = env.make_bank(clauses)
    idx = torch.arange(B, dtype=torch.int32, device="cuda")
    # int32 assignments with [B] done flags in mode 0; uint8 / bool with the reference's [B, A] flags in mode 1
    if mode == 0:
        obs_c, st_c = env.import_state(bank, idx, torch.from_numpy(assign), torch.from_numpy(step), torch.from_numpy(done))
    else:
        obs_c, st_c = env.import_state(bank, idx, torch.from_numpy(assign.astype(np.uint8)), step,
                                       np.repeat(done[:, None], env.num_agents, 1))
    assert_state_equal(st_c, st_r, "import ")
    assert np.array_equal(to_np(st_c.problem_idx), np.arange(B))
    assert_obs_equal(env._obs_dict(obs_c, True), ref.get_obs(st_r), env.agents, "import ")
    _, st_b = env.import_state(bank, idx, torch.from_numpy(assign.astype(bool)), step, done, want_obs=False)
    assert torch.equal(st_b.packed, st_c.packed)
    for t in range(3):
        acts = _actions(rng, ref, B)
        obs_r, st_r, rew_r, done_r, info_r = ref.step_env(None, st_r, acts)
        obs_c, st_c, rew_c, done_c, info_c = env.step_env(None, st_c, torch.from_numpy(acts).cuda())
        assert_obs_equal(obs_c, obs_r, env.agents, f"step {t} ")
        assert_state_equal(st_c, st_r, f"step {t} ")
        for a in env.agents:
            assert np.array_equal(to_np(rew_c[a]), rew_r[a]) and np.array_equal(to_np(done_c[a]), done_r[a])
        for key in ("solved", "num_unsatisfied", "episode_step"):
            assert np.array_equal(to_np(info_c[key]), info_r[key]), key


def test_reset_with_assignment_batched_and_unbatched():
    M = _msat()
    n, m, B = 20, 91, 5
    clauses = _formulas("uniform", B, n, m, 3, seed=3)
    assign = np.random.default_rng(0).integers(0, 2, size=(B, n)).astype(np.int32)
    ref = SATEnvOracle(n, m, 10)
    env = M.SATEnv(n, m, 10, verbose=False)
    st_r = oracle_import(ref, clauses, assign, np.zeros(B), np.zeros(B, bool))
    obs_c, st_c = env.reset_with_assignment(clauses, assign)
    assert_state_equal(st_c, st_r)
    assert_obs_equal(obs_c, ref.get_obs(st_r), env.agents)
    obs1, st1 = env.reset_with_assignment(clauses[2], assign[2], step=7, done=True)
    assert tuple(st1.variable_assignments.shape) == (n,) and int(st1.step) == 7 and bool(st1.done.all())
    for a in env.agents:
        assert np.array_equal(to_np(obs1[a]), ref.get_obs(st_r)[a][2])


# ---------------------------------------------------------------------------------------------- exact inverse
@pytest.mark.parametrize("n,m", [(20, 91), (50, 218)])
@pytest.mark.parametrize("clause_update", ["full", "incremental"])
@pytest.mark.parametrize("obs_dtype", ["int32", "int8"])
@pytest.mark.parametrize("gs", [16, 32, 64, 128, 256])
def test_reset_export_import_is_exact(gs, obs_dtype, clause_update, n, m):
    M = _msat()
    B, P = 37, 9
    env = M.SATEnv(n, m, 6, verbose=False, group_threads=gs, obs_dtype=obs_dtype, clause_update=clause_update)
    assert env._plan_for(3).dims.group_threads == gs
    bank = env.make_bank(_formulas("uniform", P, n, m, 3, seed=gs + n))
    g = torch.Generator(device="cuda").manual_seed(gs)
    idx = torch.randint(0, P, (B,), generator=g, device="cuda", dtype=torch.int32)
    keys = M.env.as_u32_tensor(_keys(B, gs + m), torch.device("cuda"))
    for want_obs in (True, False):
        obs_r, st_r = env.reset_from_bank(bank, idx, keys, want_obs=want_obs)
        obs_i, st_i = env.import_state(bank, idx, st_r.variable_assignments, want_obs=want_obs)
        assert torch.equal(st_i.packed, st_r.packed), f"packed state differs (want_obs={want_obs})"
        if want_obs:
            assert obs_i.dtype == env.obs_dtype and torch.equal(obs_i, obs_r)


@pytest.mark.parametrize("clause_update,emit_obs", [("full", True), ("incremental", False), ("incremental", True)])
def test_rollout_export_import_is_exact(clause_update, emit_obs):
    """After a de-phased rollout with auto-resets (and after stepping past done without them) the exported leaves
    import back to every packed word, including an incremental plan's per-clause counts."""
    M = _msat()
    n, m, B, P, max_steps = 50, 218, 67, 11, 5
    env = M.SATEnv(n, m, max_steps, verbose=False, clause_update=clause_update)
    bank = env.make_bank(_formulas("uniform", P, n, m, 3, seed=8))
    vec = M.VecSATEnv(env, bank, B, otf.prng_key(3), emit_obs=emit_obs)
    vec.reset()
    vec.set_episode_steps(torch.arange(B, dtype=torch.int32) % max_steps)
    g = torch.Generator(device="cuda").manual_seed(4)
    for _ in range(7):
        vec.step(torch.randint(0, 5, (B, env.num_agents), generator=g, device="cuda", dtype=torch.int32))
    st = vec.sat_state()
    obs_i, st_i = env.import_state(bank, st.problem_idx, st.variable_assignments, st.step, st.done, want_obs=emit_obs)
    assert torch.equal(st_i.packed, vec.state)
    if emit_obs:
        assert torch.equal(obs_i, vec.out["obs"])
    # past done without auto-reset: step >= max_steps and the done flag set
    cur = st_i
    for _ in range(max_steps + 2):
        _, cur, *_ = env.step_env(None, cur, torch.randint(0, 5, (B, env.num_agents), generator=g, device="cuda",
                                                           dtype=torch.int32))
    assert bool(cur.done.all()) and int(cur.step.min()) >= max_steps
    _, back = env.import_state(bank, cur.problem_idx, cur.variable_assignments, cur.step, cur.done, want_obs=False)
    assert torch.equal(back.packed, cur.packed)


def test_import_after_reset_on_a_plan_above_48k_shared_memory():
    """uf250-1065 with four groups per CTA needs the > 48 KB dynamic shared-memory opt-in; the reset makes it
    first, so the import must be covered by the same once-per-plan opt-in."""
    M = _msat()
    n, m, B, P = 250, 1065, 13, 4
    env = M.SATEnv(n, m, 16, verbose=False, group_threads=64)
    assert env._plan_for(3).dims.smem_bytes > 48 * 1024
    bank = env.make_bank(_formulas("uniform", P, n, m, 3, seed=25))
    idx = torch.arange(B, dtype=torch.int32, device="cuda") % P
    obs_r, st_r = env.reset_from_bank(bank, idx, M.env.as_u32_tensor(_keys(B, 1), torch.device("cuda")))
    obs_i, st_i = env.import_state(bank, idx, st_r.variable_assignments)
    torch.cuda.synchronize()
    assert torch.equal(st_i.packed, st_r.packed) and torch.equal(obs_i, obs_r)


def test_empty_batch_clamped_indices_and_validation():
    M = _msat()
    n, m, P = 20, 91, 6
    env = M.SATEnv(n, m, 8, verbose=False)
    bank = env.make_bank(_formulas("uniform", P, n, m, 3, seed=6))
    dev = torch.device("cuda")
    obs, st = env.import_state(bank, torch.empty(0, dtype=torch.int32), torch.empty((0, n), dtype=torch.int32))
    assert tuple(obs.shape) == (0, env.num_agents, env.obs_dim) and tuple(st.packed.shape)[0] == 0
    assign = torch.randint(0, 2, (4, n), device=dev, dtype=torch.int32)
    raw = torch.tensor([-5, 0, P + 3, P - 1], dtype=torch.int32, device=dev)
    clamped = raw.clamp(0, P - 1)
    _, st_raw = env.import_state(bank, raw, assign, validate=False)
    _, st_ok = env.import_state(bank, clamped, assign)
    assert torch.equal(st_raw.packed, st_ok.packed) and torch.equal(st_raw.problem_idx, clamped)
    with pytest.raises(IndexError):
        env.import_state(bank, raw, assign)
    bad = assign.clone()
    bad[1, 3] = 2
    with pytest.raises(ValueError, match="0 / 1"):
        env.import_state(bank, clamped, bad)
    with pytest.raises(ValueError, match="step"):
        env.import_state(bank, clamped, assign, step=torch.tensor([0, -1, 2, 3]))
    mixed = torch.zeros((4, env.num_agents), dtype=torch.bool)
    mixed[2, 0] = True
    with pytest.raises(ValueError, match="same flag"):
        env.import_state(bank, clamped, assign, done=mixed)
    with pytest.raises(ValueError):
        env.import_state(bank, clamped, assign[:, :-1])
    with pytest.raises(ValueError):
        env.import_state(bank, clamped, assign.float())


def test_vec_import_writes_the_gnn_inputs():
    M = _msat()
    n, m, B, P = 50, 218, 21, 5
    env = M.SATEnv(n, m, 8, verbose=False)
    bank = env.make_bank(_formulas("uniform", P, n, m, 3, seed=12))
    vec = M.VecSATEnv(env, bank, B, otf.prng_key(1), emit_obs=False, gnn_outputs=True)
    chain = vec.keys.chain.clone()
    assign = torch.randint(0, 2, (B, n), device="cuda", dtype=torch.int32)
    vec.import_state(torch.arange(B, dtype=torch.int32) % P, assign, torch.full((B,), 3, dtype=torch.int32))
    a_ref, cf_ref = M.dynamic_features(vec.sat_state())
    assert torch.equal(vec.out["gnn_assignment"], assign) and torch.equal(a_ref, assign)
    assert torch.equal(vec.out["gnn_clause_features"], cf_ref)
    assert torch.equal(vec.keys.chain, chain)


# ---------------------------------------------------------------------------------------------- resume / reshard
_OUT_KEYS = ("obs", "reward", "done", "solved", "num_unsatisfied", "episode_step")


def _run(vecs, actions, keys=_OUT_KEYS):
    """Step the shards of one batch with the global action table; per step the concatenated outputs."""
    rows = []
    for acts in actions:
        outs = [v.step(acts[v.env_offset:v.env_offset + v.num_envs].contiguous()) for v in vecs]
        rows.append({k: torch.cat([o[k] for o in outs]).clone() for k in keys if outs[0][k] is not None})
    return rows


def _assert_rows_equal(got, exp, what):
    for t, (g, e) in enumerate(zip(got, exp)):
        for k in g:
            assert torch.equal(g[k], e[k]), f"{what}: step {t} {k}"


def test_checkpoint_resumes_and_reshards_exactly():
    M = _msat()
    n, m, B, P, max_steps, t = 20, 91, 50, 7, 3, 5      # auto-resets in both halves
    problems = _formulas("uniform", P, n, m, 3, seed=31)
    env = M.SATEnv(n, m, max_steps, verbose=False)
    bank = env.make_bank(problems)
    key0, other = otf.prng_key(77), otf.prng_key(12345)
    g = torch.Generator(device="cuda").manual_seed(1)
    actions = [torch.randint(0, 5, (B, env.num_agents), generator=g, device="cuda", dtype=torch.int32)
               for _ in range(2 * t)]

    full = M.VecSATEnv(env, bank, B, key0)
    full.reset()
    ref_rows = _run([full], actions)
    assert any(bool(r["done"][:, -1].any()) for r in ref_rows[:t]) and any(bool(r["done"][:, -1].any()) for r in ref_rows[t:])

    first = M.VecSATEnv(env, bank, B, key0)
    first.reset()
    _assert_rows_equal(_run([first], actions[:t]), ref_rows[:t], "first half")
    sd = first.state_dict()
    assert sd["env_offset"] == 0 and sd["num_envs_global"] == B and tuple(sd["done"].shape) == (B, env.num_agents)
    obs_at_ckpt = first.out["obs"].clone()

    for world in (1, 2, 3):
        shards = [M.VecSATEnv(env, bank, B, other, world_size=world, rank=r) for r in range(world)]
        obs = torch.cat([s.load_state_dict(sd) for s in shards])
        assert torch.equal(obs, obs_at_ckpt), f"world {world}: obs after loading"
        _assert_rows_equal(_run(shards, actions[t:]), ref_rows[t:], f"world {world}")
        assert torch.equal(torch.cat([s.state for s in shards]), full.state)
        for s in shards:
            assert torch.equal(s.keys.chain, full.keys.chain)

    # rank checkpoints joined in env order load into one device
    ranks = [M.VecSATEnv(env, bank, B, other, world_size=3, rank=r) for r in range(3)]
    for s in ranks:
        s.load_state_dict(sd)
    merged = M.merge_state_dicts([s.state_dict() for s in ranks])
    single = M.VecSATEnv(env, bank, B, other)
    single.load_state_dict(merged)
    _assert_rows_equal(_run([single], actions[t:]), ref_rows[t:], "merged")
    assert torch.equal(single.state, full.state) and torch.equal(single.keys.chain, full.keys.chain)

    # a full-plan checkpoint continues on an incremental plan without observations
    env_i = M.SATEnv(n, m, max_steps, verbose=False, clause_update="incremental")
    inc = M.VecSATEnv(env_i, env_i.make_bank(problems), B, other, emit_obs=False)
    inc.load_state_dict(sd)
    _assert_rows_equal(_run([inc], actions[t:], _OUT_KEYS[1:]), ref_rows[t:], "incremental")
    a, b = inc.sat_state(), full.sat_state()
    for leaf in ("variable_assignments", "step", "done", "num_unsatisfied", "problem_idx", "clauses_satisfied_status"):
        assert torch.equal(getattr(a, leaf), getattr(b, leaf)), leaf
    assert torch.equal(inc.keys.chain, full.keys.chain)

    # mismatches are refused
    with pytest.raises(ValueError, match="signature"):
        M.VecSATEnv(env, env.make_bank(problems[:P - 1]), B, other).load_state_dict(sd)
    with pytest.raises(ValueError, match="envs"):
        M.VecSATEnv(env, bank, B + 1, other).load_state_dict(sd)
    part = ranks[1].state_dict()
    with pytest.raises(ValueError, match="cover"):
        M.VecSATEnv(env, bank, B, other, world_size=3, rank=0).load_state_dict(part)


def test_graph_captured_import_replays_to_the_eager_result():
    M = _msat()
    n, m, B, P = 50, 218, 33, 8
    env = M.SATEnv(n, m, 10, verbose=False)
    bank = env.make_bank(_formulas("uniform", P, n, m, 3, seed=44))
    dev = torch.device("cuda")
    idx = torch.zeros(B, dtype=torch.int32, device=dev)
    assign = torch.zeros((B, n), dtype=torch.int32, device=dev)
    step = torch.zeros(B, dtype=torch.int32, device=dev)
    done = torch.zeros(B, dtype=torch.uint8, device=dev)
    vec = M.VecSATEnv(env, bank, B, otf.prng_key(2))
    vec.reset()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                        # warm-up outside the capture
        vec.import_state(idx, assign, step, done, validate=False)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        vec.import_state(idx, assign, step, done, validate=False)
    g = torch.Generator(device="cuda").manual_seed(9)
    idx.copy_(torch.randint(0, P, (B,), generator=g, device=dev, dtype=torch.int32))
    assign.copy_(torch.randint(0, 2, (B, n), generator=g, device=dev, dtype=torch.int32))
    step.copy_(torch.randint(0, 20, (B,), generator=g, device=dev, dtype=torch.int32))
    done.copy_(torch.randint(0, 2, (B,), generator=g, device=dev, dtype=torch.int32).to(torch.uint8))
    vec.state.zero_()
    vec.out["obs"].zero_()
    graph.replay()
    torch.cuda.synchronize()
    eager = M.VecSATEnv(env, bank, B, otf.prng_key(2))
    eager.import_state(idx.clone(), assign.clone(), step.clone(), done.clone())
    assert torch.equal(vec.state, eager.state) and torch.equal(vec.out["obs"], eager.out["obs"])
    assert int(vec.sat_state().step.max()) > 0 and bool(vec.sat_state().done.any())
