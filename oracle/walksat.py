"""NumPy restatement of ``msat_walksat`` (batched WalkSAT/SKC, ``include/marl_sat_b200.h``), one env at a time.

Break counts are computed by brute force: the formula is re-evaluated with the variable flipped, using
``SATEnvOracle.calculate_satisfaction``.  Nothing here shares structure with the kernel (no occurrence lists, no
incremental counts).

Algorithm contract (restated word for word from the header):

The loop is per env.  Flip iteration t runs for t = 0 .. max_flips-1 and stops early as soon as num_unsat == 0;
an env that is already satisfied on entry makes 0 flips.  Each iteration does the following:
  1. Random bits.  c = flip_offset + t (uint32); (x0, x1) = threefry2x32(key[b], ctr = (c, 0)).
  2. Clause choice.  U = num_unsat, r = umulhi(x0, U).  The picked clause is the r-th unsatisfied clause
     (0-based) in increasing clause index.
  3. Candidates.  The clause's non-padding literal columns j = 0..k-1, in column order; duplicates stay in
     the list.  nc = their count.  If nc == 0 (an all-padding clause) nothing is flipped, but the iteration
     still counts.
  4. Break counts.  break(v) = the number of distinct clauses that are satisfied now and unsatisfied after
     flipping v alone: a satisfied clause breaks iff all of its true literals are on v and it has no false
     literal on v.  Literal 0 is never true (env:135-144).
  5. Choice of variable.  If some candidate has break 0, the first such candidate (freebie).  Otherwise, if
     (x1 >> 8) < thr with thr = llrint(noise * 2^24), a random walk: candidate ((x1 & 0xFF) * nc) >> 8.
     Otherwise the first candidate with the minimum break.
  6. Flip.  Flip the chosen variable and update the true-literal counts, the status and num_unsat.
A call with max_flips = F1 + F2 gives the same result, bit for bit, as a call with F1 followed by a call with
F2 and flip_offset = F1 on the returned state with the same keys.
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import numpy as np

from . import threefry
from .sat_env import SATEnvOracle, _jax_gather_index


def noise_threshold(noise: float) -> int:
    """thr = llrint(noise * 2^24) (round half to even, as llrint in the default rounding mode)."""
    return int(np.rint(np.float64(noise) * 16777216.0))


def random_bits(key, c: int) -> Tuple[int, int]:
    """(x0, x1) = threefry2x32(key, ctr = (c, 0)) for the uint32 counter c."""
    x0, x1 = threefry.threefry2x32(np.uint32(key[0]), np.uint32(key[1]), np.array([c & 0xFFFFFFFF], np.uint32),
                                   np.zeros(1, np.uint32))
    return int(x0[0]), int(x1[0])


def walksat_one(ref: SATEnvOracle, clauses: np.ndarray, assign: np.ndarray, key, max_flips: int, noise: float,
                flip_offset: int = 0, trace: Optional[List[dict]] = None) -> Tuple[np.ndarray, int, int]:
    """One env: clauses int32[m, k] (DIMACS literals, 0 = padding), assign int32[n] (0 / 1), key uint32[2].
    Returns (assignment after the search, num_unsatisfied, iterations used).  ``trace`` (optional) receives one
    dict per iteration: clause, candidates, breaks, branch ("empty" / "freebie" / "walk" / "greedy"), var."""
    n = ref.num_vars
    cl = np.asarray(clauses, np.int32)[None]
    a = (np.asarray(assign) != 0).astype(np.int32)[None].copy()
    thr = noise_threshold(noise)
    var_of = _jax_gather_index(np.abs(cl[0]) - 1, n)          # the variable a literal reads (env:135,139)
    status, nu = ref.calculate_satisfaction(a, cl)
    t = 0
    while t < max_flips and nu[0] > 0:
        x0, x1 = random_bits(key, flip_offset + t)
        U = int(nu[0])
        r = (x0 * U) >> 32                                     # umulhi(x0, U)
        c = int(np.flatnonzero(~status[0])[r])
        cols = [j for j in range(cl.shape[2]) if cl[0, c, j] != 0]
        step = {"t": t, "clause": c, "candidates": [int(var_of[c, j]) for j in cols]}
        if not cols:
            step["branch"] = "empty"
        else:
            cands = step["candidates"]
            flipped = np.repeat(a, len(cands), axis=0)
            flipped[np.arange(len(cands)), cands] ^= 1
            st_after, _ = ref.calculate_satisfaction(flipped, np.repeat(cl, len(cands), axis=0))
            breaks = [int((status[0] & ~st_after[i]).sum()) for i in range(len(cands))]
            step["breaks"] = breaks
            if 0 in breaks:
                pick, step["branch"] = breaks.index(0), "freebie"
            elif (x1 >> 8) < thr:
                pick, step["branch"] = ((x1 & 0xFF) * len(cands)) >> 8, "walk"
            else:
                pick, step["branch"] = breaks.index(min(breaks)), "greedy"
            v = cands[pick]
            step["var"] = v
            a[0, v] ^= 1
            status, nu = ref.calculate_satisfaction(a, cl)
        if trace is not None:
            trace.append(step)
        t += 1
    return a[0], int(nu[0]), t


def walksat(ref: SATEnvOracle, clauses: np.ndarray, assign: np.ndarray, keys: np.ndarray, max_flips: int,
            noise: float = 0.5, flip_offset: int = 0):
    """Batched driver: clauses int32[B, m, k], assign int32[B, n], keys uint32[B, 2].  Returns (assign int32[B, n],
    num_unsatisfied int32[B], solved bool[B], flips int32[B])."""
    clauses = np.asarray(clauses, np.int32)
    out = (np.asarray(assign) != 0).astype(np.int32).copy()
    keys = np.asarray(keys, np.uint32)
    B = out.shape[0]
    nu = ref.calculate_satisfaction(out, clauses)[1].astype(np.int32)
    flips = np.zeros(B, np.int32)
    for b in range(B):
        out[b], nu[b], flips[b] = walksat_one(ref, clauses[b], out[b], keys[b], max_flips, noise, flip_offset)
    return out, nu, nu == 0, flips
