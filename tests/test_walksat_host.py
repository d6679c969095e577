"""CPU tests of the batched WalkSAT (``msat_walksat``, ``marl_sat_b200.walksat``) and of its NumPy oracle: argument
errors are returned before anything is enqueued, the Python entry point refuses to run without a CUDA device, the
oracle follows a hand-derived trajectory through every branch of the algorithm and solves the planted reference
formulas.  No kernel is launched here."""
import ctypes as C
import math
from pathlib import Path

import numpy as np
import pytest
import torch

import marl_sat_b200 as M
from marl_sat_b200 import _lib, dimacs
from oracle.sat_env import SATEnvOracle
from oracle.walksat import noise_threshold, random_bits, walksat, walksat_one

GOLD_DIR = Path(__file__).resolve().parent / "golden"


def _aligned_buf(nbytes=4096):
    buf = (C.c_char * (nbytes + 256))()
    return buf, (C.addressof(buf) + 127) // 128 * 128


def test_walksat_argument_errors_enqueue_nothing():
    lib = _lib.load()
    env = M.SATEnv(20, 91, 8, verbose=False, device="cpu")
    plan = env._plan_for(3).handle
    keep, a = _aligned_buf()
    call = lambda plan=plan, bank=a, P=1, state=a, keys=a, F=10, off=0, noise=0.5, solved=None, flips=None, B=4: \
        lib.msat_walksat(plan, bank, P, state, keys, F, off, noise, solved, flips, B, None)
    assert call(plan=None) == _lib.MSAT_EINVAL
    assert call(P=0) == _lib.MSAT_EINVAL
    assert call(B=-1) == _lib.MSAT_EINVAL
    # missing pointers while there are envs to search
    assert call(bank=None) == _lib.MSAT_EINVAL
    assert call(state=None) == _lib.MSAT_EINVAL
    assert call(keys=None) == _lib.MSAT_EINVAL
    # noise outside [0, 1] or NaN
    for noise in (-1e-9, 1.0 + 1e-9, math.nan, math.inf):
        assert call(noise=noise) == _lib.MSAT_EINVAL, noise
    # flip budget
    assert call(F=-1) == _lib.MSAT_EINVAL
    assert call(off=-1) == _lib.MSAT_EINVAL
    assert call(F=2 ** 31 - 1, off=1) == _lib.MSAT_EINVAL
    assert call(F=2 ** 30, off=2 ** 30) == _lib.MSAT_EINVAL
    # misaligned bank / state
    assert call(bank=a + 16) == _lib.MSAT_EALIGN
    assert call(state=a + 4) == _lib.MSAT_EALIGN
    # no envs: nothing to do, nothing needed (no device is touched)
    assert call(bank=None, state=None, keys=None, B=0) == _lib.MSAT_OK
    assert call(noise=0.0, F=0, B=0) == _lib.MSAT_OK and call(noise=1.0, F=2 ** 31 - 2, off=1, B=0) == _lib.MSAT_OK
    assert "msat_walksat" in _lib.SIGNATURES


def test_walksat_unsupported_shapes():
    lib = _lib.load()
    keep, a = _aligned_buf()
    # more than 32 literal columns: one lane per candidate
    envs = []          # the envs own the plans

    def plan(n, m, k):
        envs.append(M.SATEnv(n, m, 8, verbose=False, device="cpu"))
        return envs[-1]._plan_for(k).handle

    wide = plan(40, 20, 33)
    assert lib.msat_walksat(wide, a, 1, a, a, 10, 0, 0.5, None, None, 4, None) == _lib.MSAT_EUNSUPPORTED
    # literal block + occurrence lists of one env larger than a CTA's shared memory
    big = plan(20, 32767, 2)
    assert lib.msat_walksat(big, a, 1, a, a, 10, 0, 0.5, None, None, 4, None) == _lib.MSAT_EUNSUPPORTED
    # uf250-1065 and mixed k <= 7 fit
    for n, m, k in ((250, 1065, 3), (100, 430, 7)):
        assert lib.msat_walksat(plan(n, m, k), a, 1, a, a, 10, 0, 0.5, None, None, 0, None) == _lib.MSAT_OK


def test_walksat_has_no_cpu_fallback_and_validates_on_the_host():
    env = M.SATEnv(20, 91, 8, verbose=False, device="cpu")
    state = M.SATState(env, None, torch.zeros((2, 4), dtype=torch.int32), True)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        M.walksat(state, np.zeros((2, 2), np.uint32), 10)
    assert M.WalkSATResult._fields == ("state", "solved", "flips")


def test_noise_threshold():
    assert noise_threshold(0.0) == 0 and noise_threshold(1.0) == 1 << 24 and noise_threshold(0.5) == 1 << 23
    assert noise_threshold(2.5 / 2 ** 24) == 2 and noise_threshold(3.5 / 2 ** 24) == 4    # llrint: half to even


# ------------------------------------------------------------------------------------------------ trajectory
# n = 3, key = (7, 1), noise = 0.5 (thr = 2^23), start from x = 000.  C4 is all padding (never satisfied).
TINY = np.array([[1, 2, 0],        # C0  x1 | x2
                 [-1, 2, 0],       # C1 ~x1 | x2
                 [1, -2, 0],       # C2  x1 | ~x2
                 [-1, -2, 3],      # C3 ~x1 | ~x2 | x3
                 [0, 0, 0],        # C4  (empty)
                 [-3, 1, 0],       # C5 ~x3 | x1
                 [-3, 2, 0]],      # C6 ~x3 | x2
                np.int32)


def test_oracle_follows_the_hand_derived_trajectory():
    """Derived by hand from the contract:
      t  x0          x1          unsat       r  clause  breaks      branch                     flip  after
      0  0x08f2ada3  0xd6d7ec8f  {C0,C4}     0  C0      x1:1 x2:1   greedy (x1>>8 >= 2^23)     x1    100
      1  0x6a633d33  0xe133a0ad  {C1,C4}     0  C1      x1:1 x2:1   greedy                     x1    000
      2  0x7326206f  0x06f5e6d9  {C0,C4}     0  C0      x1:1 x2:1   walk ((0xd9 * 2) >> 8 = 1) x2    010
      3  0x38e00e3a  0xf059f845  {C2,C4}     0  C2      x1:1 x2:1   greedy                     x1    110
      4  0xe7f31982  0x78082888  {C3,C4}     1  C4      -           empty clause               -     110
      5  0x6e463973  0x7a9feaf5  {C3,C4}     0  C3      x1:1 x2:1 x3:0  freebie                x3    111
    (break of x1 at t = 0: 100 falsifies C1; of x2: 010 falsifies C2; and so on.)  U = 1 (C4) after t = 5, so the
    search runs out its budget of 6 flips unsolved."""
    key = np.array([7, 1], np.uint32)
    bits = [(0x08F2ADA3, 0xD6D7EC8F), (0x6A633D33, 0xE133A0AD), (0x7326206F, 0x06F5E6D9), (0x38E00E3A, 0xF059F845),
            (0xE7F31982, 0x78082888), (0x6E463973, 0x7A9FEAF5)]
    assert [random_bits(key, t) for t in range(6)] == bits
    ref = SATEnvOracle(3, TINY.shape[0], max_steps=4)
    trace = []
    a, nu, t = walksat_one(ref, TINY, np.zeros(3, np.int32), key, 6, 0.5, trace=trace)
    got = [(s["clause"], s.get("breaks"), s["branch"], s.get("var")) for s in trace]
    assert got == [(0, [1, 1], "greedy", 0), (1, [1, 1], "greedy", 0), (0, [1, 1], "walk", 1),
                   (2, [1, 1], "greedy", 0), (4, None, "empty", None), (3, [1, 1, 0], "freebie", 2)]
    assert a.tolist() == [1, 1, 1] and nu == 1 and t == 6
    # resumable: 4 + 2 flips with flip_offset = 4 equal 6 flips
    a4, _, t4 = walksat_one(ref, TINY, np.zeros(3, np.int32), key, 4, 0.5)
    a6, nu6, t6 = walksat_one(ref, TINY, a4, key, 2, 0.5, flip_offset=4)
    assert (a6.tolist(), nu6, t4 + t6) == ([1, 1, 1], 1, 6)
    # noise 0 never walks, noise 1 always walks unless there is a freebie
    for noise, banned in ((0.0, "walk"), (1.0, "greedy")):
        tr = []
        walksat_one(ref, TINY, np.zeros(3, np.int32), key, 40, noise, trace=tr)
        assert banned not in {s["branch"] for s in tr}


def test_oracle_solves_the_planted_reference_formulas():
    files = sorted(GOLD_DIR.glob("ref_*.cnf"))
    assert len(files) == 8
    for i, path in enumerate(files):
        n, m, clauses = dimacs.parse_cnf_native(str(path))
        ref = SATEnvOracle(n, clauses.shape[0], max_steps=4)
        key = np.array([[0, i]], np.uint32)
        assign, nu, solved, flips = walksat(ref, clauses[None], np.zeros((1, n), np.int32), key, 20000, 0.5)
        assert solved[0] and nu[0] == 0, path.name
        assert ref.calculate_satisfaction(assign, clauses[None])[0].all(), path.name
        # already satisfied on entry: no flips, nothing changes
        again = walksat(ref, clauses[None], assign, key, 100, 0.5)
        assert again[3][0] == 0 and np.array_equal(again[0], assign)
