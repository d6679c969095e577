"""GPU tests of the on-device action draw (``msat_sample_actions``): parity with the NumPy oracle over class counts
and shards, bit-identical sharding, the key pinned to the reference fixtures' act_keys, the softmax distribution,
exact resume / reshard of a sampled rollout, CUDA-graph capture and the MAPPO trainer's act-key path."""
import copy

import numpy as np
import pytest
import torch

from oracle import rollout as orollout
from oracle import sampling as osamp
from oracle import threefry as otf
from tests.test_golden_env import ROLLOUT_CASES, load

pytestmark = pytest.mark.gpu


def _msat():
    import marl_sat_b200 as M
    return M


def _oracle_scores(key, logits):
    """float64 scores g + z and log-softmax z of every row (the oracle's intermediate values)."""
    C = logits.shape[-1]
    l = np.asarray(logits, np.float32).reshape(-1, C).astype(np.float64)
    _, u = osamp.uniform_bits(key, l.size)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        sh = l - l.max(1, keepdims=True)
        z = sh - np.log(np.exp(sh).sum(1, keepdims=True))
        return osamp.gumbel(u).reshape(l.shape) + z, z


def _assert_oracle_draw(actions, log_prob, key, logits, rows=None):
    """Device draw == oracle draw wherever the best score leads by more than 1e-4 * max(1, |best|), else one of the
    top two; at least 99.9 % of rows exact; log_prob within 1e-6 relative + 1e-6 absolute of the oracle's z of the
    drawn class.  ``rows`` selects global rows of ``logits`` that the device outputs hold (default: all)."""
    C = logits.shape[-1]
    a, lp, margin = (x.reshape(-1) for x in osamp.categorical(key, logits))
    score, z = _oracle_scores(key, logits)
    if rows is not None:
        a, lp, margin, score, z = a[rows], lp[rows], margin[rows], score[rows], z[rows]
    ga = actions.reshape(-1).cpu().numpy()
    glp = log_prob.reshape(-1).cpu().numpy().astype(np.float64)
    assert ga.shape == a.shape
    idx = np.arange(a.size)
    valid = a >= 0
    best = np.where(valid, score[idx, np.maximum(a, 0)], 0.0)
    clear = margin > 1e-4 * np.maximum(1.0, np.abs(best))
    assert np.array_equal(ga[clear], a[clear]), f"{int((ga[clear] != a[clear]).sum())} clear draws differ"
    near = ~clear
    if near.any():
        top2 = np.argsort(-score[near], axis=1, kind="stable")[:, :2]
        assert ((ga[near] == top2[:, 0]) | (ga[near] == top2[:, 1])).all(), "a near tie outside the top two"
    assert (ga == a).mean() >= 0.999
    assert np.isneginf(glp[~valid]).all()
    want = z[idx[valid], ga[valid]]
    assert np.allclose(glp[valid], want, rtol=1e-6, atol=1e-6), f"max log_prob err {np.abs(glp[valid] - want).max()}"


def _logits(shape, seed, scale=2.5):
    return (np.random.default_rng(seed).normal(size=shape) * scale).astype(np.float32)


@pytest.mark.parametrize("C", [1, 2, 5, 9, 18, 33, 64])
@pytest.mark.parametrize("rows_global", [1000, 1001])
def test_oracle_parity(C, rows_global):
    M = _msat()
    logits = _logits((rows_global, C), seed=C * 7 + rows_global)
    if C > 1:        # -inf entries in valid rows and every kind of invalid row
        logits[::11, C // 2] = -np.inf
        logits[5, C - 1] = np.nan
        logits[17, 0] = np.inf
        logits[29, :] = -np.inf
        logits[41, :] = -np.inf
        logits[41, C - 1] = 1.0
    key_rng = otf.prng_key(77 + C)
    key = osamp.act_key(key_rng)
    dev_logits = torch.from_numpy(logits).cuda()
    rng = torch.from_numpy(key_rng.view(np.int32)).cuda()
    a, lp = M.sample_actions(dev_logits, rng)
    torch.cuda.synchronize()
    _assert_oracle_draw(a, lp, key, logits)
    if C > 1:
        assert a[5].item() == a[17].item() == a[29].item() == -1 and a[41].item() == C - 1
    # an uneven shard of the same global table
    off, rows = 137, 700
    a_s, lp_s = M.sample_actions(dev_logits[off:off + rows], rng, num_rows_global=rows_global, row_offset=off)
    _assert_oracle_draw(a_s, lp_s, key, logits, rows=np.arange(off, off + rows))
    assert torch.equal(a_s, a[off:off + rows]) and torch.equal(lp_s, lp[off:off + rows])


def test_oracle_parity_at_the_headline_shape():
    """65,536 envs x 25 agents x 5 classes (uf100-430, mode 0): every 509th row against the oracle."""
    M = _msat()
    shape = (65536, 25, 5)
    logits = _logits(shape, seed=509, scale=1.5)
    key_rng = otf.prng_key(2026)
    a, lp = M.sample_actions(torch.from_numpy(logits).cuda(), torch.from_numpy(key_rng.view(np.int32)).cuda())
    assert a.shape == lp.shape == shape[:2]
    rows = np.arange(0, 65536 * 25, 509)
    _assert_oracle_draw(a.reshape(-1)[torch.from_numpy(rows).cuda()], lp.reshape(-1)[torch.from_numpy(rows).cuda()],
                        osamp.act_key(key_rng), logits.reshape(-1, 5), rows=rows)


@pytest.mark.parametrize("C", [5, 33])
def test_shard_invariance(C):
    M = _msat()
    rows_global = 5003
    logits = torch.from_numpy(_logits((rows_global, C), seed=C)).cuda()
    rng = torch.tensor([12345, -6789], dtype=torch.int32, device="cuda")
    a1, lp1 = M.sample_actions(logits, rng)
    cut_rng = np.random.default_rng(C)
    for shards in (1, 2, 3, 7):
        cuts = [0] + sorted(cut_rng.choice(np.arange(1, rows_global), shards - 1, replace=False).tolist()) + [rows_global]
        parts = [M.sample_actions(logits[lo:hi], rng, num_rows_global=rows_global, row_offset=lo)
                 for lo, hi in zip(cuts[:-1], cuts[1:])]
        assert torch.equal(torch.cat([p[0] for p in parts]), a1), (shards, cuts)
        assert torch.equal(torch.cat([p[1] for p in parts]), lp1), (shards, cuts)


@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("name", ROLLOUT_CASES)
def test_key_is_the_reference_act_key(name, weighted):
    """Before each step of a fixture's rollout, ``vec.sample_actions`` draws with the act_key the unmodified reference
    passed to ``pi.sample`` (the fixture's ``act_keys``), in both action modes and while problem weights are set."""
    M = _msat()
    fx = load(name)
    c = fx["cfg"]
    T, B = c["T"], c["B"]
    env = M.SATEnv(c["n"], c["m"], c["max_steps"], vars_per_agent=c["vpa"], action_mode=c["mode"], verbose=False,
                   **fx["reward_kw"])
    vec = M.VecSATEnv(env, torch.from_numpy(fx["clauses"]), B, fx["key0"])
    if weighted:
        vec.set_problem_weights(np.arange(1, c["P"] + 1))
    vec.reset()
    A, V = env.num_agents, env.max_vars_per_agent
    shape = (B, A, V + 1) if c["mode"] == 0 else (B, A, V, 2)
    actions = torch.from_numpy(fx["actions"]).cuda()
    for t in range(T):
        logits = _logits(shape, seed=1000 * t + 17)
        a, lp = vec.sample_actions(torch.from_numpy(logits).cuda())
        assert a.shape == shape[:-1] and lp.shape == shape[:-1]
        _assert_oracle_draw(a, lp, fx["act_keys"][t], logits)
        vec.step(actions[t])


def test_draws_follow_the_softmax():
    """One logits row repeated over 2^20 rows: the class counts pass a chi-square test against its softmax (the rng
    is fixed, so the test is deterministic)."""
    from scipy import stats
    M = _msat()
    row = torch.tensor([0.3, -1.2, 2.0, 0.0, -0.5, 1.1, -3.0, 0.7, -0.1], dtype=torch.float32)
    n = 2 ** 20
    logits = row.expand(n, row.numel()).contiguous().cuda()
    a, lp = M.sample_actions(logits, torch.tensor([3, 1415926], dtype=torch.int32, device="cuda"))
    counts = torch.bincount(a.long(), minlength=row.numel()).cpu().numpy()
    p = torch.softmax(row.double(), 0).numpy()
    assert counts.sum() == n and stats.chisquare(counts, p * n).pvalue > 1e-3
    assert torch.allclose(lp.double(), torch.log_softmax(row.double(), 0).cuda()[a.long()], rtol=1e-6, atol=1e-6)


# ---------------------------------------------------------------------------------------------------------------
# sampled rollouts: resume / reshard, graph capture
# ---------------------------------------------------------------------------------------------------------------
def _env_and_bank(M, max_steps=5):
    from marl_sat_b200.synth import uniform_ksat
    env = M.SATEnv(50, 218, max_steps, verbose=False)
    return env, env.make_bank(uniform_ksat(8, 50, 218, 3, seed=41))


def _policy_logits(vec):
    """Logits that are elementwise functions of each env's own observation (no matmul: shard-invariant)."""
    obs = vec.out["obs"]
    V = vec.env.max_vars_per_agent
    return obs[:, :, :V + 1].float() * 1.5 + obs[:, :, V + 1:2 * V + 2].float() * 0.25


def _sampled_steps(shards, steps):
    """``steps`` sampled rollout steps on every shard; per step the shard outputs concatenated in env order."""
    rec = []
    for _ in range(steps):
        row = {k: [] for k in ("action", "log_prob", "reward", "done", "solved", "num_unsatisfied", "episode_step")}
        for vec in shards:
            a, lp = vec.sample_actions(_policy_logits(vec))
            out = vec.step(a)
            row["action"].append(a.clone())
            row["log_prob"].append(lp.clone())
            for k in ("reward", "done", "solved", "num_unsatisfied", "episode_step"):
                row[k].append(out[k].clone())
        rec.append({k: torch.cat(v) for k, v in row.items()})
    return rec


def test_resume_and_reshard_continue_the_uninterrupted_rollout():
    M = _msat()
    env, bank = _env_and_bank(M)
    B, key = 96, otf.prng_key(3)
    full = M.VecSATEnv(env, bank, B, key)
    full.reset()
    ref = _sampled_steps([full], 12)
    assert any(bool(r["done"].any()) for r in ref)              # episodes end and auto-reset inside the window
    first = M.VecSATEnv(env, bank, B, key)
    first.reset()
    head = _sampled_steps([first], 6)
    sd = first.state_dict()
    for world in (2, 3):
        shards = [M.VecSATEnv(env, bank, B, key, world_size=world, rank=r) for r in range(world)]
        for s in shards:
            s.load_state_dict(sd)
        tail = _sampled_steps(shards, 6)
        for t, rec in enumerate(head + tail):
            for k, v in rec.items():
                assert torch.equal(v, ref[t][k]), f"world {world}: step {t} {k}"
        assert torch.equal(torch.cat([s.state for s in shards]), full.state), f"world {world}: final state"
        assert torch.equal(torch.cat([s.out["obs"] for s in shards]), full.out["obs"]), f"world {world}: final obs"
        for s in shards:
            assert torch.equal(s.keys.chain, full.keys.chain)


def test_graph_capture_replays_to_the_eager_result():
    M = _msat()
    env, bank = _env_and_bank(M)
    B, G, key = 256, 2, otf.prng_key(8)
    graphed, eager = M.VecSATEnv(env, bank, B, key), M.VecSATEnv(env, bank, B, key)
    graphed.reset()
    eager.reset()
    A, V = env.num_agents, env.max_vars_per_agent
    acts = torch.empty((G, B, A), dtype=torch.int32, device="cuda")
    lps = torch.empty((G, B, A), dtype=torch.float32, device="cuda")
    logits = torch.empty((B, A, V + 1), dtype=torch.float32, device="cuda")

    def steps():
        for t in range(G):
            logits.copy_(_policy_logits(graphed))
            graphed.sample_actions(logits, acts[t], lps[t])
            graphed.step(acts[t])

    saved = (graphed.state.clone(), graphed.keys._bufs.clone(), graphed.keys._cur, graphed.out["obs"].clone())

    def restore():
        graphed.state.copy_(saved[0])
        graphed.keys._bufs.copy_(saved[1])
        graphed.keys._cur = saved[2]
        graphed.out["obs"].copy_(saved[3])

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                   # warm-up outside the capture, then put the env back
        steps()
    torch.cuda.current_stream().wait_stream(side)
    restore()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        steps()
    restore()
    acts.zero_()
    lps.zero_()
    graph.replay()
    ref = _sampled_steps([eager], G)
    torch.cuda.synchronize()
    for t in range(G):
        assert torch.equal(acts[t], ref[t]["action"]) and torch.equal(lps[t], ref[t]["log_prob"]), t
    assert torch.equal(graphed.state, eager.state) and torch.equal(graphed.out["obs"], eager.out["obs"])


def test_trainer_draws_with_the_act_key():
    """``MAPPOTrainer(act_key_sampling=True)``: every stored action is the oracle draw with that step's act_key on the
    logits of the pre-update network, recomputed from the stored pre-step observations (autocast off)."""
    M = _msat()
    from marl_sat_b200.mappo import MAPPOTrainer, MLPActorCritic, PPOConfig
    from marl_sat_b200.synth import uniform_ksat
    env = M.SATEnv(20, 91, 6, verbose=False)
    bank = env.make_bank(uniform_ksat(16, 20, 91, 3, seed=2))
    B, T = 64, 5
    vec = M.VecSATEnv(env, bank, B, otf.prng_key(11))
    vec.reset()
    torch.manual_seed(0)
    net = MLPActorCritic(env, hidden=32)
    trainer = MAPPOTrainer(vec, net, PPOConfig(num_steps=T, update_epochs=1, minibatch_size=64), autocast=False,
                           act_key_sampling=True)
    before = copy.deepcopy(trainer.raw_net)
    rng = M.env.u32_to_numpy(vec.keys.rng).copy()
    metrics = trainer.train_cycle()
    assert metrics["optimizer_steps"] > 0
    buf = trainer.buf
    for t in range(T):
        ks = orollout.rollout_keys(rng, B, bank.num_problems)
        rng = ks["rng"]
        with torch.no_grad():
            logits = before.actor_logits(buf.local_obs(t)).cpu().numpy()
        a, lp = buf.action[t], buf.log_prob[t]
        _assert_oracle_draw(a, lp, ks["act_key"], logits)
