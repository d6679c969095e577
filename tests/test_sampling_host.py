"""CPU tests of the on-device action draw (``msat_sample_actions``, ``marl_sat_b200.sample_actions``,
``VecSATEnv.sample_actions``) and of its NumPy oracle: argument errors are returned before anything is enqueued,
the Python entry points validate their tensors and refuse CPU tensors, and the oracle has the properties the
contract states (exact bits, finite Gumbel values, the reference's act_key, -inf entries never drawn, invalid rows,
the softmax distribution).  No kernel is launched here."""
import ctypes as C
import types

import numpy as np
import pytest
import torch
from scipy import stats

import marl_sat_b200 as M
from marl_sat_b200 import _lib
from oracle import rollout as orollout
from oracle import sampling as osamp
from oracle import threefry as otf


def test_sample_actions_argument_errors_enqueue_nothing():
    lib = _lib.load()
    buf = (C.c_float * 256)()
    a = (C.addressof(buf) + 15) // 16 * 16

    def call(logits=a, Bg=10, off=0, rows=4, ncls=5, rng=a, actions=a, log_prob=a):
        return lib.msat_sample_actions(logits, Bg, off, rows, ncls, rng, actions, log_prob, None)
    # missing pointers while there are rows to draw
    assert call(logits=None) == _lib.MSAT_EINVAL
    assert call(rng=None) == _lib.MSAT_EINVAL
    assert call(actions=None) == _lib.MSAT_EINVAL
    # class count, negative counts / offsets, rows outside the global table
    assert call(ncls=0) == _lib.MSAT_EINVAL and call(ncls=-3) == _lib.MSAT_EINVAL
    assert call(rows=-1) == _lib.MSAT_EINVAL
    assert call(Bg=-1) == _lib.MSAT_EINVAL
    assert call(off=-1) == _lib.MSAT_EINVAL
    assert call(off=7) == _lib.MSAT_EINVAL and call(Bg=3) == _lib.MSAT_EINVAL
    assert call(off=2 ** 62, Bg=2 ** 62) == _lib.MSAT_EINVAL
    # alignment of the float buffers
    assert call(logits=a + 2) == _lib.MSAT_EALIGN
    assert call(log_prob=a + 1) == _lib.MSAT_EALIGN
    # N = num_rows_global * C must stay below 2^32 - 1 (JAX's single-block counter path)
    assert call(Bg=(2 ** 32 - 1) // 5 + 1) == _lib.MSAT_EUNSUPPORTED
    assert call(Bg=2 ** 32 - 1, ncls=1) == _lib.MSAT_EUNSUPPORTED
    assert call(Bg=2 ** 40, ncls=2 ** 30) == _lib.MSAT_EUNSUPPORTED
    # no rows: nothing to do, nothing needed (no device is touched)
    assert call(logits=None, rng=None, actions=None, log_prob=None, rows=0) == _lib.MSAT_OK
    assert call(logits=None, rng=None, actions=None, log_prob=None, rows=0, Bg=0, off=0) == _lib.MSAT_OK
    assert "msat_sample_actions" in _lib.SIGNATURES


def test_python_validation_raises_without_enqueueing():
    logits = torch.zeros((4, 3, 5), dtype=torch.float32)
    rng = np.array([0, 42], np.uint32)
    with pytest.raises(ValueError, match="float32"):
        M.sample_actions(logits.double(), rng)
    with pytest.raises(ValueError, match="float32"):
        M.sample_actions(logits.numpy(), rng)
    with pytest.raises(ValueError, match="C >= 1"):
        M.sample_actions(torch.zeros((4, 0)), rng)
    with pytest.raises(ValueError, match="C >= 1"):
        M.sample_actions(torch.zeros(()), rng)
    with pytest.raises(ValueError, match="contiguous"):
        M.sample_actions(logits.transpose(0, 1), rng)
    with pytest.raises(ValueError, match="outside the global table"):
        M.sample_actions(logits, rng, num_rows_global=11)
    with pytest.raises(ValueError, match="outside the global table"):
        M.sample_actions(logits, rng, num_rows_global=20, row_offset=9)
    with pytest.raises(ValueError, match="outside the global table"):
        M.sample_actions(logits, rng, row_offset=-1, num_rows_global=20)
    with pytest.raises(ValueError, match="2\\*\\*32"):
        M.sample_actions(logits, rng, num_rows_global=2 ** 31)
    with pytest.raises(ValueError, match="CUDA"):
        M.sample_actions(logits, rng)


def _fake_vec(mode, B=4, A=3, V=7):
    env = types.SimpleNamespace(num_agents=A, max_vars_per_agent=V, action_mode=mode)
    return types.SimpleNamespace(env=env, num_envs=B, state=types.SimpleNamespace(device=torch.device("cuda", 0)))


@pytest.mark.parametrize("mode", [0, 1])
def test_vec_env_checks_the_logits_shape_and_device(mode):
    vec = _fake_vec(mode)
    good = (4, 3, 8) if mode == 0 else (4, 3, 7, 2)
    bad = [(4, 3, 7), (4, 3, 7, 2) if mode == 0 else (4, 3, 8), (3,) + good[1:], (12,) + good[2:]]
    for shape in bad:
        with pytest.raises(ValueError, match="logits must be"):
            M.VecSATEnv.sample_actions(vec, torch.zeros(shape))
    with pytest.raises(ValueError, match="logits must be"):
        M.VecSATEnv.sample_actions(vec, np.zeros(good, np.float32))
    with pytest.raises(ValueError, match="cuda"):
        M.VecSATEnv.sample_actions(vec, torch.zeros(good))


# ---------------------------------------------------------------------------------------------------------------
# oracle properties
# ---------------------------------------------------------------------------------------------------------------
def test_oracle_bits_are_the_threefry_stream():
    key = otf.prng_key(11)
    for n in (1, 2, 7, 1000, 1001):
        bits, u = osamp.uniform_bits(key, n)
        assert np.array_equal(bits, otf.random_bits32(key, n))
        f = ((bits >> np.uint32(9)) | np.uint32(0x3F800000)).view(np.float32) - np.float32(1)
        assert u.dtype == np.float32 and np.array_equal(u, np.where(f == 0, np.finfo(np.float32).tiny, f))
        assert (u > 0).all() and (u < 1).all()


def test_oracle_gumbel_is_finite_at_both_ends():
    tiny = np.finfo(np.float32).tiny
    top = np.float32(1) - np.float32(2.0 ** -23)                 # the largest uniform: f = 1 - 2^-23
    f0 = np.float32(0)
    u0 = np.maximum(np.float32(tiny), f0 * (np.float32(1) - np.float32(tiny)) + np.float32(tiny))
    assert u0 == np.float32(tiny)                                 # f = 0 maps to FLT_MIN
    g = osamp.gumbel(np.array([u0, top], np.float32))
    assert np.isfinite(g).all() and g[0] < -4 and g[1] > 15


def test_oracle_act_key_is_the_reference_chain_key():
    # SURVEY.md App. B: one learner step from rng = PRNGKey(42) draws act_key = [255383827, 267815257]
    assert osamp.act_key(otf.prng_key(42)).tolist() == [255383827, 267815257]
    rng = otf.prng_key(1234)
    for _ in range(4):
        ks = orollout.rollout_keys(rng, 8, 3)
        assert np.array_equal(osamp.act_key(rng), ks["act_key"])
        rng = ks["rng"]


def test_oracle_never_draws_minus_inf_and_flags_invalid_rows():
    rng = np.random.default_rng(3)
    logits = rng.normal(size=(4000, 6)).astype(np.float32)
    logits[:, 1] = -np.inf
    logits[::3, 4] = -np.inf
    a, lp, margin = osamp.categorical(otf.prng_key(5), logits)
    assert (a != 1).all() and (a[::3] != 4).all() and np.isfinite(lp).all() and (lp <= 0).all()
    assert (margin >= 0).all()
    bad = np.zeros((6, 4), np.float32)
    bad[0, 2] = np.nan
    bad[1, 0] = np.inf
    bad[2, :] = -np.inf
    bad[3, :] = [np.nan, np.inf, -np.inf, 0]
    bad[4, :] = [-np.inf, -np.inf, 3.0, -np.inf]                  # one finite entry: always drawn, log_prob 0
    a, lp, margin = osamp.categorical(otf.prng_key(6), bad)
    assert a[:4].tolist() == [-1] * 4 and np.isneginf(lp[:4]).all()
    assert a[4] == 2 and lp[4] == 0.0 and 0 <= a[5] < 4
    # one class: always class 0 with log_prob 0
    a, lp, _ = osamp.categorical(otf.prng_key(7), np.full((5, 1), 3.5, np.float32))
    assert (a == 0).all() and (lp == 0).all()


def test_oracle_log_prob_is_the_log_softmax_of_the_draw():
    rng = np.random.default_rng(4)
    logits = (rng.normal(size=(3, 50, 9)) * 4).astype(np.float32)
    a, lp, _ = osamp.categorical(otf.prng_key(8), logits)
    assert a.shape == lp.shape == (3, 50)
    l64 = logits.astype(np.float64)
    ref = l64 - l64.max(-1, keepdims=True)
    ref = ref - np.log(np.exp(ref).sum(-1, keepdims=True))
    assert np.allclose(lp, np.take_along_axis(ref, a[..., None].astype(np.int64), -1)[..., 0], rtol=0, atol=1e-12)


def test_oracle_draws_follow_the_softmax():
    """10^5 rows of one logits vector: the class counts pass a chi-square test against its softmax."""
    row = np.array([0.3, -1.2, 2.0, 0.0, -0.5, 1.1, -3.0], np.float32)
    n = 100_000
    a, _, _ = osamp.categorical(otf.prng_key(2024), np.broadcast_to(row, (n, row.size)))
    p = np.exp(row.astype(np.float64) - row.max())
    p /= p.sum()
    counts = np.bincount(a, minlength=row.size)
    assert stats.chisquare(counts, p * n).pvalue > 1e-3
