"""CPU tests of the state import (msat_import_state) and the rollout checkpoints: argument errors are returned
before anything is enqueued, the Python entry points refuse to run without a CUDA device, and checkpoints of
adjacent shards merge in env order.  No kernel is launched here."""
import ctypes as C

import numpy as np
import pytest
import torch

import marl_sat_b200 as M
from marl_sat_b200 import _lib


def _aligned_buf(nbytes=4096):
    buf = (C.c_char * (nbytes + 256))()
    return buf, (C.addressof(buf) + 127) // 128 * 128


def test_import_state_argument_errors_enqueue_nothing():
    lib = _lib.load()
    env = M.SATEnv(20, 91, 8, verbose=False, device="cpu")
    plan = env._plan_for(3).handle
    keep, a = _aligned_buf()
    call = lambda plan=plan, bank=a, P=1, idx=a, va=a, step=None, done=None, state=a, obs=None, B=4: \
        lib.msat_import_state(plan, bank, P, idx, va, step, done, state, obs, B, None)
    assert call(plan=None) == _lib.MSAT_EINVAL
    assert call(P=0) == _lib.MSAT_EINVAL
    assert call(B=-1) == _lib.MSAT_EINVAL
    # a required pointer missing while there are envs to import
    assert call(bank=None) == _lib.MSAT_EINVAL
    assert call(idx=None) == _lib.MSAT_EINVAL
    assert call(va=None) == _lib.MSAT_EINVAL
    assert call(state=None) == _lib.MSAT_EINVAL
    # misaligned outputs / bank
    assert call(state=a + 4) == _lib.MSAT_EALIGN
    assert call(obs=a + 8) == _lib.MSAT_EALIGN
    assert call(bank=a + 16) == _lib.MSAT_EALIGN
    # no envs: nothing to do, nothing needed (no device is touched)
    assert call(bank=None, idx=None, va=None, state=None, B=0) == _lib.MSAT_OK
    assert "msat_import_state" in _lib.SIGNATURES


def test_import_entry_points_have_no_cpu_fallback():
    env = M.SATEnv(20, 91, 8, verbose=False, device="cpu")
    clauses = np.ones((91, 3), np.int32)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        env.reset_with_assignment(clauses, np.zeros(20, np.int32))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        env.import_state(None, torch.zeros(1, dtype=torch.int32), torch.zeros((1, 20), dtype=torch.int32))


def _ckpt(offset, rows, chain=0, n=4, A=2, num_envs_global=10):
    return {"variable_assignments": torch.arange(offset, offset + rows, dtype=torch.int32)[:, None].repeat(1, n),
            "step": torch.arange(offset, offset + rows, dtype=torch.int32),
            "done": torch.zeros((rows, A), dtype=torch.bool),
            "problem_idx": torch.arange(offset, offset + rows, dtype=torch.int32),
            "rng_chain": torch.full((10,), chain, dtype=torch.int32),
            "env_offset": offset, "num_envs_global": num_envs_global,
            "signature": {"num_vars": n, "num_clauses": 3, "k": 3, "num_agents": A, "num_problems": 5}}


def test_merge_state_dicts_joins_adjacent_shards_in_env_order():
    parts = [_ckpt(*M.shard_range(10, 3, r)) for r in range(3)]
    merged = M.merge_state_dicts(parts[::-1])
    assert merged["env_offset"] == 0 and merged["num_envs_global"] == 10
    assert merged["step"].tolist() == list(range(10))
    assert merged["variable_assignments"].shape == (10, 4) and merged["done"].shape == (10, 2)
    assert torch.equal(merged["rng_chain"], parts[0]["rng_chain"])
    # the tail of a run only (rows 3..9) is a valid checkpoint of those rows
    assert M.merge_state_dicts(parts[1:])["env_offset"] == parts[1]["env_offset"]
    with pytest.raises(ValueError, match="adjacent"):
        M.merge_state_dicts([parts[0], parts[2]])
    with pytest.raises(ValueError, match="rng chains differ"):
        M.merge_state_dicts([parts[0], _ckpt(parts[1]["env_offset"], 3, chain=1)])
    with pytest.raises(ValueError, match="different runs"):
        M.merge_state_dicts([parts[0], _ckpt(parts[1]["env_offset"], 3, num_envs_global=11)])
