"""CPU tests of the curriculum primitives: argument errors of ``msat_env_keys_weighted`` / ``msat_problem_stats`` are
returned before anything is enqueued, ``problem_weights`` validates and quantises, and the NumPy oracle's weighted
draw and per-problem statistics have the properties the contract promises.  No kernel is launched here."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import marl_sat_b200 as M
from marl_sat_b200 import _lib
from oracle import curriculum as ocur
from oracle import features as ofeat
from oracle import threefry as otf


def _aligned_buf(nbytes=4096):
    buf = (C.c_char * (nbytes + 256))()
    return buf, (C.addressof(buf) + 127) // 128 * 128


def test_env_keys_weighted_argument_errors_enqueue_nothing():
    lib = _lib.load()
    keep, a = _aligned_buf()
    call = lambda pk=a, rk=a, Bg=64, off=0, Bl=16, cum=a, P=7, idx=a, keys=a: \
        lib.msat_env_keys_weighted(pk, rk, Bg, off, Bl, cum, P, idx, keys, None)
    # missing pointers while there are envs to draw for
    assert call(pk=None) == _lib.MSAT_EINVAL
    assert call(cum=None) == _lib.MSAT_EINVAL
    assert call(rk=None) == _lib.MSAT_EINVAL
    # problem count and shard
    for P in (0, -1):
        assert call(P=P) == _lib.MSAT_EINVAL
    assert call(off=60, Bl=16) == _lib.MSAT_EINVAL          # shard beyond the batch
    assert call(off=-1) == _lib.MSAT_EINVAL and call(Bl=-1) == _lib.MSAT_EINVAL and call(Bg=-1) == _lib.MSAT_EINVAL
    assert call(Bg=(1 << 30) + 1, Bl=16) == _lib.MSAT_EUNSUPPORTED
    # int64 prefix sums must be 8-byte aligned
    assert call(cum=a + 4) == _lib.MSAT_EALIGN
    # empty shard: nothing to do, nothing enqueued (no device is touched)
    assert call(Bl=0) == _lib.MSAT_OK and call(off=64, Bl=0) == _lib.MSAT_OK
    assert "msat_env_keys_weighted" in _lib.SIGNATURES


def test_problem_stats_argument_errors_enqueue_nothing():
    lib = _lib.load()
    keep, a = _aligned_buf()
    call = lambda pidx=a, st=4, sb=1, done=a, sol=a, nu=a, es=a, T=3, B=4, P=5, stats=a: \
        lib.msat_problem_stats(pidx, st, sb, done, sol, nu, es, T, B, P, stats, None)
    for name in ("pidx", "done", "sol", "nu", "es"):
        assert call(**{name: None}) == _lib.MSAT_EINVAL, name
    assert call(stats=None) == _lib.MSAT_EINVAL and call(stats=None, T=0) == _lib.MSAT_EINVAL
    for P in (0, -3):
        assert call(P=P) == _lib.MSAT_EINVAL
    assert call(T=-1) == _lib.MSAT_EINVAL and call(B=-1) == _lib.MSAT_EINVAL
    assert call(stats=a + 4) == _lib.MSAT_EALIGN
    # no rows: nothing read, nothing enqueued
    assert call(pidx=None, done=None, sol=None, nu=None, es=None, T=0) == _lib.MSAT_OK
    assert call(pidx=None, done=None, sol=None, nu=None, es=None, B=0) == _lib.MSAT_OK
    assert "msat_problem_stats" in _lib.SIGNATURES


def test_problem_stats_has_no_cpu_fallback():
    z = torch.zeros((2, 3), dtype=torch.int32)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        M.problem_stats(z, z.to(torch.uint8), z.to(torch.uint8), z, z, 4)


def test_problem_weights_validation_and_quantisation():
    q = M.problem_weights([0.0, 1.0, 0.5, 2.0])
    # (2^32 - 1) / 2 = 2^31 - 0.5 rounds half to even: 2^31; (2^32 - 1) / 4 = 2^30 - 0.25 rounds to 2^30
    assert q.dtype == torch.int64 and q.tolist() == [0, 2 ** 31, 2 ** 30, 2 ** 32 - 1]
    assert q.tolist() == ocur.quantize_weights([0.0, 1.0, 0.5, 2.0]).tolist()
    assert M.problem_weights(torch.tensor([True, False, True])).tolist() == [2 ** 32 - 1, 0, 2 ** 32 - 1]
    assert M.problem_weights(np.array([3, 3, 3], np.int32)).tolist() == [2 ** 32 - 1] * 3
    assert M.problem_weights([1e-300, 1.0]).tolist() == [0, 2 ** 32 - 1]        # tiny weights may round to 0
    assert M.problem_weights([5.0], num_problems=1).tolist() == [2 ** 32 - 1]
    bad = [([[1.0, 2.0]], "shape"), (np.ones(3), "shape"), ([1.0, math.nan], "finite"), ([1.0, math.inf], "finite"),
           ([1.0, -1e-9], "non-negative"), ([0.0, 0.0], "all zero"), (np.array(["a", "b"]), "real")]
    for w, match in bad:
        with pytest.raises(ValueError, match=match):
            M.problem_weights(w, num_problems=2)
    with pytest.raises(ValueError, match="shape"):
        M.problem_weights([])


def test_unsolved_weights():
    stats = torch.tensor([[10, 10, 0, 50], [10, 3, 9, 4], [0, 0, 0, 0], [4, 0, 8, 0]], dtype=torch.int64)
    w = M.unsolved_weights(stats)
    assert w.dtype == torch.float64 and w.tolist() == [0.1, 0.7, 1.0, 1.0]
    assert M.unsolved_weights(stats, floor=0.0).tolist() == [0.0, 0.7, 1.0, 1.0]
    with pytest.raises(ValueError):
        M.unsolved_weights(stats[:, :3])


# ------------------------------------------------------------------------------------------------ oracle draw
def test_oracle_zero_weight_problem_is_never_drawn():
    cum = np.cumsum([5, 0, 0, 7, 0, 1, 0], dtype=np.int64)
    for seed in range(4):
        idx = ocur.weighted_randint(otf.prng_key(seed), 5000, cum)
        assert set(np.unique(idx).tolist()) <= {0, 3, 5}
        assert set(np.unique(idx).tolist()) == {0, 3, 5}


def test_oracle_zero_total_falls_back_to_randint():
    for P in (1, 7, 800):
        for cum in (np.zeros(P, np.int64), np.full(P, -3, np.int64)):
            assert np.array_equal(ocur.weighted_randint(otf.prng_key(P), 1001, cum), otf.randint(otf.prng_key(P), 1001, 0, P))


def test_oracle_non_monotone_table_stays_in_range():
    cum = np.array([9, 2, 2 ** 40, -5, 3, 2 ** 40 + 1], np.int64)
    idx = ocur.weighted_randint(otf.prng_key(3), 4000, cum)
    assert idx.min() >= 0 and idx.max() < len(cum)


def test_oracle_draw_follows_the_weights_chi_square():
    from scipy import stats as sps
    w = np.array([1.0, 0.0, 3.0, 0.25, 7.0, 2.0, 0.5])
    q = ocur.quantize_weights(w)
    N = 10 ** 6
    idx = ocur.weighted_randint(otf.prng_key(2026), N, np.cumsum(q))
    counts = np.bincount(idx, minlength=len(w))
    assert counts[1] == 0
    keep = q > 0
    expected = q[keep] / q[keep].sum() * N
    chi2, pval = sps.chisquare(counts[keep], expected)
    assert pval > 1e-4, (chi2, pval, counts)


# ------------------------------------------------------------------------------------------------ oracle stats
def test_oracle_stats_sum_to_the_rollout_metrics():
    rng = np.random.default_rng(7)
    T, B, P = 40, 300, 13
    done = rng.random((T, B)) < 0.2
    solved = rng.random((T, B)) < 0.5
    nu = rng.integers(0, 50, (T, B)).astype(np.int32) * ~solved
    es = rng.integers(1, 30, (T, B)).astype(np.int32)
    pidx = rng.integers(-2, P + 2, (T, B)).astype(np.int32)
    reward = (solved & done).astype(np.float32)
    stats = ocur.problem_stats(pidx, done, solved, nu, es, P)
    assert stats.shape == (P, 4) and stats.dtype == np.int64
    tot = stats.sum(axis=0)
    met = ofeat.rollout_metrics(reward, done, solved, nu, es)
    assert tot[0] == done.sum() and tot[0] > 0
    assert met["solve_rate"] == float(tot[1] / max(tot[0], 1.0))
    assert met["avg_unsatisfied_clauses"] == float(tot[2] / max(tot[0], 1.0))
    assert met["avg_steps_to_solve"] == float(tot[3] / max(tot[1], 1.0))
    # clamping: the out-of-range indices land on the first and last rows
    low, high = done & (pidx <= 0), done & (pidx >= P - 1)
    assert stats[0, 0] == low.sum() and stats[P - 1, 0] == high.sum()
