"""CPU tests of the start states (``msat_apply_start_states``): argument errors are returned before anything is
enqueued, ``start_table`` validates, packs and quantises, ``adapt_flip_prob`` follows its rule, and the NumPy oracle's
start draw has the properties the contract promises.  No kernel is launched here."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import marl_sat_b200 as M
from marl_sat_b200 import _lib
from marl_sat_b200.curriculum import adapt_flip_prob, flip_thresholds, start_table
from oracle import start_states as ostart
from oracle import threefry as otf
from oracle.sat_env import SATEnvOracle


def _aligned_buf(nbytes=4096):
    buf = (C.c_char * (nbytes + 256))()
    return buf, (C.addressof(buf) + 127) // 128 * 128


def test_apply_start_states_argument_errors_enqueue_nothing():
    lib = _lib.load()
    env = M.SATEnv(20, 91, 8, verbose=False, device="cpu")
    plan = env._plan_for(3).handle
    keep, a = _aligned_buf()
    call = lambda plan=plan, bank=a, P=5, st=a, rk=a, Bg=64, off=0, words=a, thr=a, has=a, obs=a, ga=None, gc=None, \
        B=16: lib.msat_apply_start_states(plan, bank, P, st, rk, Bg, off, words, thr, has, obs, ga, gc, B, None)
    # missing pointers while there are envs
    for name in ("plan", "bank", "st", "rk", "words", "thr"):
        assert call(**{name: None}) == _lib.MSAT_EINVAL, name
    # counts and shard
    for P in (0, -1):
        assert call(P=P) == _lib.MSAT_EINVAL
    assert call(B=-1) == _lib.MSAT_EINVAL and call(Bg=-1) == _lib.MSAT_EINVAL and call(off=-1) == _lib.MSAT_EINVAL
    assert call(off=60, B=16) == _lib.MSAT_EINVAL                    # shard beyond the batch
    assert call(Bg=(1 << 30) + 1) == _lib.MSAT_EUNSUPPORTED
    # alignment: bank 128, state / obs 16, tables and GNN outputs 4
    assert call(bank=a + 16) == _lib.MSAT_EALIGN and call(st=a + 4) == _lib.MSAT_EALIGN
    assert call(obs=a + 4) == _lib.MSAT_EALIGN
    assert call(words=a + 2) == _lib.MSAT_EALIGN and call(thr=a + 1) == _lib.MSAT_EALIGN
    assert call(ga=a + 2) == _lib.MSAT_EALIGN and call(gc=a + 2) == _lib.MSAT_EALIGN
    # no envs: nothing read, nothing enqueued (no device is touched); has_start / outputs are optional
    assert call(B=0) == _lib.MSAT_OK and call(off=64, B=0) == _lib.MSAT_OK
    assert call(bank=None, st=None, rk=None, words=None, thr=None, has=None, obs=None, B=0) == _lib.MSAT_OK
    assert "msat_apply_start_states" in _lib.SIGNATURES


def test_flip_thresholds_quantisation_and_validation():
    assert flip_thresholds(0.0, 3).tolist() == [0, 0, 0]
    assert flip_thresholds(0.5, 1).tolist() == [2 ** 31]
    assert flip_thresholds(1.0, 2).tolist() == [2 ** 32 - 1] * 2
    q = [0.0, 0.25, 0.5, 1.0, 2.0 ** -33, 3 * 2.0 ** -33, 0.05]
    t = flip_thresholds(q, len(q))
    assert t.dtype == torch.int64
    # round half to even: 0.5 -> 0, 1.5 -> 2
    assert t.tolist() == [0, 2 ** 30, 2 ** 31, 2 ** 32 - 1, 0, 2, round(0.05 * 2 ** 32)]
    assert t.tolist() == ostart.quantize_flip_prob(q).tolist()
    assert flip_thresholds(torch.tensor([1, 0]), 2).tolist() == [2 ** 32 - 1, 0]
    for bad, match in (([0.1, math.nan], "finite"), ([0.1, math.inf], "finite"), ([0.1, 1.0 + 1e-9], r"\[0, 1\]"),
                       ([-1e-12, 0.0], r"\[0, 1\]"), (np.ones(3), "shape"), (np.array(["a", "b"]), "real")):
        with pytest.raises(ValueError, match=match):
            flip_thresholds(bad, 2)


def test_start_table_packing_bit_order_and_flags():
    n = 70                                          # three words, the last one partial
    a = np.zeros((3, n), np.int32)
    a[0, [0, 31, 32, 69]] = 1
    a[1] = 1
    a[2, 5] = 7                                     # nonzero reads as 1
    a[2, 64] = -1
    t = start_table(a, [0.0, 0.5, 1.0], has_start=[1, 0, 5])
    assert t.words.dtype == torch.int32 and tuple(t.words.shape) == (3, 3)
    words = t.words.numpy().view(np.uint32)
    assert words[0].tolist() == [1 | (1 << 31), 1, 1 << 5]
    assert words[1].tolist() == [2 ** 32 - 1, 2 ** 32 - 1, (1 << 6) - 1]       # bits past n stay 0
    assert words[2].tolist() == [1 << 5, 0, 1]
    assert np.array_equal(words, ostart.pack_assignments(a))
    assert t.flip_thr.tolist() == [0, 2 ** 31, 2 ** 32 - 1]
    assert t.has_start.dtype == torch.uint8 and t.has_start.tolist() == [1, 0, 1]
    assert start_table(torch.ones((2, 5), dtype=torch.bool), 0.25).has_start.tolist() == [1, 1]
    assert start_table(a, 0.1).flip_thr.tolist() == [round(0.1 * 2 ** 32)] * 3
    for bad, match in ((np.zeros((4,), np.int32), "shape"), (np.zeros((0, 5), np.int32), "shape"),
                       (np.zeros((2, 5), np.float32), "integers or booleans")):
        with pytest.raises(ValueError, match=match):
            start_table(bad, 0.0)
    with pytest.raises(ValueError, match="has_start"):
        start_table(a, 0.0, has_start=[1, 1])
    with pytest.raises(ValueError, match="has_start"):
        start_table(a, 0.0, has_start=[0.5, 1.0, 0.0])
    with pytest.raises(ValueError, match="flip_prob"):
        start_table(a, [0.1, 0.2])


def test_adapt_flip_prob_rule():
    # finished, solved: rates 1.0, 0.9 (>= high), 0.5 (between), 0.2 (<= low), 0.0, and no finished episode
    stats = torch.tensor([[10, 10, 0, 5], [10, 9, 1, 5], [10, 5, 9, 5], [10, 2, 9, 5], [4, 0, 9, 0], [0, 0, 0, 0]],
                         dtype=torch.int64)
    q = [0.1, 0.4, 0.1, 0.1, 0.011, 0.3]
    out = adapt_flip_prob(stats, q, low=0.2, high=0.8, factor=2.0, q_min=0.01, q_max=0.5)
    assert out.dtype == torch.float64 and tuple(out.shape) == (6,)
    assert out.tolist() == pytest.approx([0.2, 0.5, 0.1, 0.05, 0.01, 0.3], rel=0, abs=1e-15)
    # a scalar q, q = 0 grows through the floor, and the untouched problem keeps an out-of-range-of-clamp value
    out = adapt_flip_prob(stats, 0.0, factor=1.5, q_min=0.02, q_max=0.5)
    assert out.tolist() == [0.02, 0.02, 0.02, 0.02, 0.02, 0.0]
    with pytest.raises(ValueError):
        adapt_flip_prob(stats[:, :3], q)
    with pytest.raises(ValueError):
        adapt_flip_prob(stats, q, q_min=0.6, q_max=0.5)
    with pytest.raises(ValueError):
        adapt_flip_prob(stats, q, factor=0.5)
    with pytest.raises(ValueError):
        adapt_flip_prob(stats, [0.1, 2.0, 0.1, 0.1, 0.1, 0.1])


# ------------------------------------------------------------------------------------------------ oracle
def _env_keys(seed, B):
    return otf.split(otf.prng_key(seed), B)


def test_oracle_threshold_zero_is_the_start_and_the_maximum_its_complement():
    rng = np.random.default_rng(0)
    for n in (1, 20, 33, 100, 251):
        P, B = 5, 400
        start = rng.integers(0, 2, (P, n)).astype(np.int32)
        p = rng.integers(0, P, B)
        keys = _env_keys(n, B)
        assert np.array_equal(ostart.start_assignments(start, np.zeros(P, np.int64), p, keys), start[p])
        # u < 2^32 - 1 fails only for u = 2^32 - 1 (probability 2^-32 per bit); these keys never draw it
        assert (ostart.flip_words(keys, n) != 2 ** 32 - 1).all()
        assert np.array_equal(ostart.start_assignments(start, np.full(P, 2 ** 32 - 1, np.int64), p, keys), 1 - start[p])


def test_oracle_flip_words_are_randint_layout_under_ka():
    """u_v = threefry_2x32(ka, arange(n))[v]: the same counter layout as randint's draw, under the other half of
    split(K); bit 0 of the draw under kb is the reset's assignment."""
    keys = _env_keys(3, 64)
    for n in (7, 8, 100):
        u = ostart.flip_words(keys, n)
        for b in (0, 17, 63):
            ka, kb = otf.split(keys[b])
            assert np.array_equal(u[b], otf.random_bits32(ka, n))
            assert np.array_equal(otf.random_bits32(kb, n) & 1, otf.randint01_many(keys[b:b + 1], n)[0])


def test_oracle_flips_are_independent_of_the_random_draw():
    """Under one key, the flip mask at q = 1/2 and randint's assignment bits are independent: a 2x2 contingency
    chi-square over 10^5 x 100 bit pairs, and the joint cell frequencies near 1/4."""
    from scipy import stats as sps
    B, n = 100_000, 100
    keys = _env_keys(2026, B)
    flips = ostart.flip_words(keys, n) < np.uint32(2 ** 31)
    draw = otf.randint01_many(keys, n) != 0
    table = np.array([[np.sum(~flips & ~draw), np.sum(~flips & draw)], [np.sum(flips & ~draw), np.sum(flips & draw)]])
    chi2, pval, _, _ = sps.chi2_contingency(table, correction=False)
    assert pval > 1e-4, (chi2, pval, table)
    assert np.abs(table / table.sum() - 0.25).max() < 0.002
    # and per variable: neither the flip rate nor its agreement with the draw depends on v
    assert np.abs(flips.mean(axis=0) - 0.5).max() < 0.01
    assert np.abs((flips == draw).mean(axis=0) - 0.5).max() < 0.01


@pytest.mark.parametrize("q", [0.05, 0.5])
def test_oracle_hamming_distance_is_binomial(q):
    """Over 10^5 draws the Hamming distance to the start has the mean and variance of Binomial(n, thr / 2^32)
    within 5-sigma bounds of the sample mean and variance."""
    B, n, P = 100_000, 100, 3
    start = np.random.default_rng(1).integers(0, 2, (P, n)).astype(np.int32)
    thr = ostart.quantize_flip_prob(np.full(P, q))
    p = np.arange(B) % P
    x = ostart.start_assignments(start, thr, p, _env_keys(int(q * 1000), B))
    dist = (x != start[p]).sum(axis=1).astype(np.float64)
    pr = thr[0] / 2.0 ** 32
    mu, var = n * pr, n * pr * (1 - pr)
    mu4 = var * (1 + 3 * (n - 2) * pr * (1 - pr))              # fourth central moment of the binomial
    assert abs(dist.mean() - mu) < 5 * math.sqrt(var / B), (dist.mean(), mu)
    assert abs(dist.var(ddof=1) - var) < 5 * math.sqrt((mu4 - var * var * (B - 3) / (B - 1)) / B), (dist.var(), var)


def test_oracle_apply_selects_restarted_envs_with_a_start():
    from marl_sat_b200.synth import uniform_ksat
    n, m, P, B = 20, 91, 4, 12
    problems = uniform_ksat(P, n, m, 3, seed=3)
    ref = SATEnvOracle(n, m, 5)
    idx = np.arange(B) % P
    keys = _env_keys(9, B)
    obs, st = ref.reset(problems[idx], keys)
    obs = np.stack([obs[a] for a in ref.agents], 1)
    st = st.__class__(**{**st.__dict__, "step": np.where(np.arange(B) % 3 == 0, 1, 0).astype(np.int32)})
    start = np.random.default_rng(2).integers(0, 2, (P, n)).astype(np.int32)
    has = np.array([1, 1, 0, 1])
    new, nobs = ostart.apply_start_states(ref, st, obs, idx, keys, (start, np.zeros(P, np.int64), has))
    sel = (st.step == 0) & (has[idx] != 0)
    assert sel.any() and (~sel).any()
    assert np.array_equal(new.variable_assignments[sel], start[idx[sel]])
    assert np.array_equal(new.variable_assignments[~sel], st.variable_assignments[~sel])
    assert np.array_equal(nobs[~sel], obs[~sel])
    status, nu = ref.calculate_satisfaction(new.variable_assignments, new.clauses)
    assert np.array_equal(new.num_unsatisfied, nu) and np.array_equal(new.clauses_satisfied_status, status)
    assert np.array_equal(nobs[sel], ref.get_obs_array(new)[sel])
