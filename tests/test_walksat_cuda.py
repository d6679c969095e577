"""GPU tests of the batched WalkSAT (``msat_walksat``, ``marl_sat_b200.walksat``).

* oracle parity: for every parity shape, both clause-update modes and noise 0 / 0.5 / 1 the kernel matches
  ``oracle/walksat.py`` in every packed state word, in ``solved`` and in ``flips``; also at uf100-430 x 65,536;
* solutions: every env reported solved satisfies every clause (planted reference formulas, loose uf50-150);
* continuation, nothing-to-do, interop with ``get_obs`` / the exported leaves, and graph capture.
"""
import numpy as np
import pytest
import torch

from oracle.sat_env import SATEnvOracle
from oracle.walksat import walksat as oracle_walksat
from tests.test_parity_cuda import SHAPES
from tests.test_state_import_cuda import _formulas, _keys, oracle_import
from tests.util import STATE_LEAVES, assert_obs_equal, to_np

pytestmark = pytest.mark.gpu


def _msat():
    import marl_sat_b200 as M
    return M


def _reset(env, clauses, seed):
    """Bank of the formulas and one reset env per formula."""
    bank = env.make_bank(torch.from_numpy(clauses))
    B = clauses.shape[0]
    idx = torch.arange(B, dtype=torch.int32, device="cuda")
    _, state = env.reset_from_bank(bank, idx, torch.from_numpy(_keys(B, seed).view(np.int32)).cuda(), want_obs=False)
    return bank, state


def _expected_packed(env, bank, problem_idx, assign, step=None, done=None):
    """The packed record of an assignment as the state import builds it (num_unsatisfied and counts recomputed)."""
    _, st = env.import_state(bank, problem_idx, torch.from_numpy(np.ascontiguousarray(assign, np.int32)), step, done,
                             want_obs=False)
    return to_np(st.packed)


@pytest.mark.parametrize("noise", [0.0, 0.5, 1.0])
@pytest.mark.parametrize("name,n,m,k,vpa,kind", SHAPES, ids=[s[0] for s in SHAPES])
def test_walksat_matches_oracle(name, n, m, k, vpa, kind, noise):
    M = _msat()
    B = 6 if n < 200 else 3
    F = 200
    clauses = _formulas(kind, B, n, m, k, seed=n * 3 + m)
    ref = SATEnvOracle(n, m, max_steps=8, vars_per_agent=vpa)
    keys = _keys(B, seed=m + 5)
    expected = None
    for mode in ("full", "incremental"):
        env = M.SATEnv(n, m, 8, vars_per_agent=vpa, verbose=False, clause_update=mode)
        bank, state = _reset(env, clauses, seed=n)
        before = to_np(state.packed).copy()
        if expected is None:
            start = to_np(state.variable_assignments)
            expected = oracle_walksat(ref, clauses, start, keys, F, noise)
        res = M.walksat(state, keys, F, noise=noise)
        assert np.array_equal(to_np(state.packed), before), "the input state must not change"
        idx = torch.arange(B, dtype=torch.int32)
        exp_packed = _expected_packed(env, bank, idx, expected[0])
        assert np.array_equal(to_np(res.state.packed), exp_packed), f"{mode}: packed state words differ"
        assert np.array_equal(to_np(res.solved), expected[2]), f"{mode}: solved differs"
        assert np.array_equal(to_np(res.flips), expected[3]), f"{mode}: flips differ"


def _cnf_bank_problems():
    from marl_sat_b200 import dimacs
    from pathlib import Path
    for path in sorted((Path(__file__).resolve().parent / "golden").glob("ref_*.cnf")):
        n, _, clauses = dimacs.parse_cnf_native(str(path))
        yield path.name, n, clauses[None]


def test_solved_envs_satisfy_every_clause():
    M = _msat()
    from marl_sat_b200.synth import uniform_ksat
    cases = list(_cnf_bank_problems()) + [("loose uf50-150", 50, uniform_ksat(16, 50, 150, 3, seed=11))]
    for name, n, problems in cases:
        m = problems.shape[1]
        env = M.SATEnv(n, m, 8, verbose=False)
        ref = SATEnvOracle(n, m, max_steps=8)
        B = 64
        bank = env.make_bank(torch.from_numpy(problems))
        idx = torch.arange(B, dtype=torch.int32, device="cuda") % bank.num_problems
        _, state = env.reset_from_bank(bank, idx, torch.from_numpy(_keys(B, 3).view(np.int32)).cuda(), want_obs=False)
        res = M.walksat(state, _keys(B, 4), 20000)
        solved = to_np(res.solved)
        assert solved.any(), name
        if name.startswith("ref_"):
            assert solved.all(), f"{name}: WalkSAT left a planted formula unsolved in 20,000 flips"
        nu = to_np(res.state.num_unsatisfied)
        assign = to_np(res.state.variable_assignments)
        assert np.array_equal(nu == 0, solved), name
        sat, _ = ref.calculate_satisfaction(assign[solved], problems[to_np(idx)][solved])
        assert sat.all(), f"{name}: a reported solution falsifies a clause"


def test_two_chunks_equal_one_call():
    M = _msat()
    from marl_sat_b200.synth import uniform_ksat
    for mode in ("full", "incremental"):
        env = M.SATEnv(100, 430, 8, verbose=False, clause_update=mode)
        bank, state = _reset(env, uniform_ksat(256, 100, 430, 3, seed=2), seed=9)
        keys = _keys(256, 10)
        one = M.walksat(state, keys, 1000, noise=0.5)
        a = M.walksat(state, keys, 377, noise=0.5)
        b = M.walksat(a.state, keys, 623, noise=0.5, flip_offset=377)
        assert torch.equal(one.state.packed, b.state.packed)
        assert torch.equal(one.solved, b.solved)
        assert torch.equal(one.flips, a.flips + b.flips)
        assert 0 < int(one.solved.sum()) < 256       # both solved and unsolved envs are exercised


def test_nothing_to_do_leaves_every_word():
    M = _msat()
    from marl_sat_b200.synth import uniform_ksat
    for mode in ("full", "incremental"):
        env = M.SATEnv(50, 150, 8, verbose=False, clause_update=mode)
        bank, state = _reset(env, uniform_ksat(64, 50, 150, 3, seed=4), seed=1)
        keys = _keys(64, 2)
        zero = M.walksat(state, keys, 0)
        assert torch.equal(zero.state.packed, state.packed) and not zero.flips.any()
        solved = M.walksat(state, keys, 20000)
        ok = solved.solved
        assert int(ok.sum()) >= 60
        again = M.walksat(solved.state, _keys(64, 3), 1000, noise=1.0)
        assert torch.equal(again.state.packed[ok], solved.state.packed[ok])
        assert not again.flips[ok].any() and bool(again.solved[ok].all())


@pytest.mark.parametrize("obs_dtype", ["int32", "int8"])
def test_interop_with_observations_and_leaves(obs_dtype):
    M = _msat()
    from marl_sat_b200.synth import uniform_ksat
    n, m, B, P = 100, 430, 48, 7
    problems = uniform_ksat(P, n, m, 3, seed=8)
    env = M.SATEnv(n, m, 16, verbose=False, obs_dtype=obs_dtype)
    ref = SATEnvOracle(n, m, max_steps=16)
    bank = env.make_bank(torch.from_numpy(problems))
    rng = np.random.default_rng(0)
    idx = rng.integers(0, P, B).astype(np.int32)
    assign0 = rng.integers(0, 2, (B, n)).astype(np.int32)
    step = rng.integers(0, 40, B).astype(np.int32)
    done = rng.integers(0, 2, B).astype(bool)
    _, state = env.import_state(bank, torch.from_numpy(idx), torch.from_numpy(assign0), torch.from_numpy(step),
                                torch.from_numpy(done), want_obs=False)
    res = M.walksat(state, _keys(B, 6), 500)
    new_assign = to_np(res.state.variable_assignments)
    exp = oracle_import(ref, problems[idx], new_assign, step, done)
    for leaf in STATE_LEAVES:
        got, want = to_np(getattr(res.state, leaf)), np.asarray(getattr(exp, leaf))
        assert np.array_equal(got.astype(want.dtype), want), leaf
    assert np.array_equal(to_np(res.state.problem_idx), idx)
    obs = env.get_obs(res.state)
    exp_obs = ref.get_obs(exp)
    if obs_dtype == "int32":
        assert_obs_equal(obs, exp_obs, env.agents)
    else:
        for a in env.agents:
            assert np.array_equal(to_np(obs[a]).astype(np.int32), exp_obs[a])


def test_graph_capture_replays_to_the_eager_result():
    M = _msat()
    from marl_sat_b200.synth import uniform_ksat
    env = M.SATEnv(100, 430, 8, verbose=False, clause_update="incremental")
    bank, state = _reset(env, uniform_ksat(512, 100, 430, 3, seed=5), seed=6)
    keys = torch.from_numpy(_keys(512, 7).view(np.int32)).cuda()
    eager = M.walksat(state, keys, 800)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        M.walksat(state, keys, 800)          # warm-up (and the one-time shared-memory opt-in) outside the capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        captured = M.walksat(state, keys, 800)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(captured.state.packed, eager.state.packed)
    assert torch.equal(captured.solved, eager.solved) and torch.equal(captured.flips, eager.flips)


def test_oracle_parity_at_scale():
    """uf100-430 x 65,536 envs (one formula each), 1,000 flips: every 509th env against the oracle."""
    M = _msat()
    from marl_sat_b200.synth import uniform_ksat
    n, m, B = 100, 430, 65536
    clauses = uniform_ksat(B, n, m, 3, seed=12)
    env = M.SATEnv(n, m, 8, verbose=False)
    bank, state = _reset(env, clauses, seed=13)
    keys = _keys(B, 14)
    res = M.walksat(state, keys, 1000)
    rows = np.arange(0, B, 509)
    start = to_np(state.variable_assignments)[rows]
    exp_assign, exp_nu, exp_solved, exp_flips = oracle_walksat(SATEnvOracle(n, m, max_steps=8), clauses[rows], start,
                                                               keys[rows], 1000, 0.5)
    packed = to_np(res.state.packed)[rows]
    exp_packed = _expected_packed(env, bank, torch.from_numpy(rows.astype(np.int32)), exp_assign)
    assert np.array_equal(packed, exp_packed)
    assert np.array_equal(to_np(res.solved)[rows], exp_solved)
    assert np.array_equal(to_np(res.flips)[rows], exp_flips)
