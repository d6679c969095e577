"""Drop-in ``SATEnv`` backed by the sm_100a kernels of libmarlsat_b200.so.

Mirrors the public surface of the reference environment
(``/root/reference/src/envs/multi_agent_sat_env.py``, cited as env:LINE): same constructor, same
attributes (``agents``, ``agent_groups``, ``agent_vars``, ``action_mask``, ``max_vars_per_agent``,
``variable_to_agent_idx``, ``action_spaces``, ``observation_spaces`` ...), same methods (``reset``,
``step_env``, ``get_obs``, ``action_space``, ``observation_space``, ``name``) with the same argument
meaning.  Differences that follow from being B200-native rather than a JAX program:

* the env is **natively batched**: where the reference is wrapped in ``jax.vmap`` (runner:137,
  learner:418) this class takes a leading ``B`` axis directly (unbatched calls are accepted too and
  return unbatched leaves);
* arrays are ``torch`` CUDA tensors (device memory + streams only; all arithmetic happens in the
  hand-written kernels);
* ``SATState`` keeps the packed device record (32 bytes/env at uf100-430) and materialises the
  reference-shaped leaves lazily through ``msat_export_state``;
* there is no CPU path: every compute call needs a CUDA device and the built library.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, List, Optional, Tuple, Union

import numpy as np
import torch

from . import _lib, spaces

ArrayLike = Union[np.ndarray, torch.Tensor]


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def as_u32_tensor(x: ArrayLike, device: torch.device) -> torch.Tensor:
    """uint32 payload (PRNG keys) carried in an int32 tensor with the same bits."""
    if isinstance(x, torch.Tensor):
        if x.dtype == torch.int32:
            t = x
        elif x.dtype == torch.uint32:
            t = x.view(torch.int32)
        else:
            v = x.to(torch.int64) & 0xFFFFFFFF
            t = torch.where(v >= 2 ** 31, v - 2 ** 32, v).to(torch.int32)
        return t.to(device).contiguous()
    a = np.ascontiguousarray(np.asarray(x).astype(np.uint32, copy=False)).view(np.int32)
    return torch.from_numpy(a.copy()).to(device)


def u32_to_numpy(t: torch.Tensor) -> np.ndarray:
    return t.detach().cpu().contiguous().numpy().view(np.uint32)


_OBS_POOLS: Dict[int, Optional["torch.cuda.MemPool"]] = {}


def _obs_pool(device: torch.device) -> Optional["torch.cuda.MemPool"]:
    """The device's pool of compressible memory (``msat_obs_alloc``), or None where the driver does not grant
    generic compression.  Created on first use and kept for the life of the process."""
    index = device.index if device.index is not None else torch.cuda.current_device()
    if index not in _OBS_POOLS:
        lib, granted = _lib.load(), C.c_int(0)
        _lib.check(lib.msat_obs_compression(index, C.byref(granted)), "msat_obs_compression")
        pool = None
        if granted.value:
            alloc = torch.cuda.memory.CUDAPluggableAllocator(str(_lib.lib_path()), "msat_obs_alloc", "msat_obs_free")
            pool = torch.cuda.MemPool(alloc.allocator())
        _OBS_POOLS[index] = pool
    return _OBS_POOLS[index]


def obs_empty(shape, dtype: torch.dtype, device: torch.device) -> torch.Tensor:
    """``torch.empty`` for observation buffers.  Observations (-1 / 0 / 1 words) are most of a step's DRAM
    writes; where the device grants generic compression they live in compressible memory, which DRAM stores in
    fewer bytes.  Contents and every operation on the tensor are the same either way."""
    pool = _obs_pool(device)
    if pool is None:
        return torch.empty(shape, dtype=dtype, device=device)
    with torch.cuda.use_mem_pool(pool, device):
        return torch.empty(shape, dtype=dtype, device=device)


def create_agent_groups(num_vars: int, vars_per_agent: Optional[int], verbose: bool = True) -> Dict[str, List[int]]:
    """Reference grouping rule (env:294-338): ceil(n/vpa) agents when ``vars_per_agent`` is given, else
    n/4 agents if 4 divides n, else max(2, floor(sqrt(n))); contiguous ranges, the first ``n % A``
    groups one variable larger."""
    lib = _lib.load()
    if vars_per_agent is not None:
        if verbose:
            print(f"User specified mode: aiming for {vars_per_agent} vars per agent.")
        num_agents = lib.msat_num_agents_for(num_vars, int(vars_per_agent))
    else:
        if verbose:
            print("Auto-distribution mode: Environment is determining the optimal grouping.")
        num_agents = lib.msat_num_agents_for(num_vars, 0)
        if verbose and num_vars % 4 == 0:
            print(f"Found ideal grouping: {num_agents} agents, each with 4 vars.")
    if num_agents <= 0:
        raise ValueError(f"invalid num_vars={num_vars} / vars_per_agent={vars_per_agent}")
    base, rem = divmod(num_vars, num_agents)
    groups, cur = {}, 0
    for i in range(num_agents):
        size = base + 1 if i < rem else base
        groups[f"agent_{i}"] = list(range(cur, cur + size))
        cur += size
    return groups


class _Plan:
    """RAII holder of an ``msat_plan*``."""

    def __init__(self, n, m, k, A, action_mode, max_steps, group_threads=0, reward=None, incremental=False,
                 obs_int8=False):
        self._lib = _lib.load()
        h = C.c_void_p()
        _lib.check(self._lib.msat_plan_create(C.byref(h), n, m, k, A, action_mode, max_steps, group_threads),
                   "msat_plan_create")
        self.handle = h
        if reward is not None:      # (mode, gamma, r_clause, r_sat)
            _lib.check(self._lib.msat_plan_set_reward(h, *reward), "msat_plan_set_reward")
        if incremental:             # before any bank / state is sized from the dims
            _lib.check(self._lib.msat_plan_set_clause_update(h, 1), "msat_plan_set_clause_update")
        if obs_int8:
            _lib.check(self._lib.msat_plan_set_obs_dtype(h, 1), "msat_plan_set_obs_dtype")
        self.dims = _lib.Dims()
        _lib.check(self._lib.msat_plan_dims(h, C.byref(self.dims)), "msat_plan_dims")

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self._lib.msat_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class FormulaBank:
    """P CNF formulas compiled into HBM-resident records (packed literals + flat agent-mask stream).

    Replaces ``problems['clauses']`` (runner:118) as the thing the rollout draws new episodes from.
    """

    def __init__(self, env: "SATEnv", clauses: ArrayLike, validate: bool = True):
        cl = clauses if isinstance(clauses, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(clauses))
        if cl.dim() != 3 or cl.shape[1] != env.num_clauses:
            raise ValueError(f"clauses must be [P, {env.num_clauses}, k], got {tuple(cl.shape)}")
        device = env._require_cuda()
        cl = cl.to(device=device, dtype=torch.int32).contiguous()
        if validate and cl.numel() and int(cl.abs().max()) > env.num_vars:
            raise ValueError("a literal refers to a variable index > num_vars")
        self.env = env
        self.num_problems = int(cl.shape[0])
        self.k = int(cl.shape[2])
        self.plan = env._plan_for(self.k)
        self.clauses = cl
        self.data = torch.empty(max(1, self.num_problems) * self.plan.dims.rec_bytes, dtype=torch.uint8, device=device)
        _lib.check(env._lib.msat_compile_bank(self.plan.handle, _ptr(cl), self.num_problems, _ptr(self.data),
                                              _stream_ptr(device)), "msat_compile_bank")


    def for_env(self, env: "SATEnv") -> "FormulaBank":
        """The same compiled records bound to another env object of the same shape and grouping (e.g. a
        different ``max_steps`` or reward variant): the record layout depends only on (n, m, k, A)."""
        d0, plan = self.plan.dims, env._plan_for(self.k)
        d1 = plan.dims
        if (d0.n, d0.m, d0.k, d0.A, d0.rec_bytes) != (d1.n, d1.m, d1.k, d1.A, d1.rec_bytes):
            raise ValueError("for_env needs an env with the same (n, m, k, agents)")
        other = object.__new__(FormulaBank)
        other.__dict__.update(self.__dict__)
        other.env, other.plan = env, plan
        return other


class SATState:
    """Mirror of the reference ``SATState`` (env:13-24) plus the jaxmarl ``State`` fields
    (``done``, ``step``).  Holds the packed per-env device record; the reference-shaped leaves
    are exported on first access (and cached)."""

    _LEAVES = ("variable_assignments", "clauses_satisfied_status", "num_unsatisfied", "step", "done", "clauses",
               "agent_clause_masks", "agent_neighbor_masks", "literal_to_agent_idx")

    def __init__(self, env: "SATEnv", bank: FormulaBank, packed: torch.Tensor, batched: bool):
        self.env, self.bank, self.packed, self.batched = env, bank, packed, batched
        self._cache: Dict[str, torch.Tensor] = {}

    @property
    def num_envs(self) -> int:
        return int(self.packed.shape[0])

    @property
    def action_mask(self) -> torch.Tensor:
        return self.env.action_mask

    @property
    def problem_idx(self) -> torch.Tensor:
        return self._leaf("problem_idx")

    def _leaf(self, name: str) -> torch.Tensor:
        if name not in self._cache:
            self._export(name)
        t = self._cache[name]
        return t if self.batched else t[0]

    # leaf -> (shape builder, dtype); exported one at a time so that reading `step` does not
    # materialise the [B, A, m] masks
    _EXPORT_ORDER = ("variable_assignments", "clauses_satisfied_status", "num_unsatisfied", "step", "done", "clauses",
                     "agent_clause_masks", "agent_neighbor_masks", "literal_to_agent_idx", "problem_idx")

    def _export(self, name: str) -> None:
        env, d = self.env, self.bank.plan.dims
        B, dev = self.num_envs, self.packed.device
        shapes = {
            "variable_assignments": ((B, d.n), torch.int32), "clauses_satisfied_status": ((B, d.m), torch.uint8),
            "num_unsatisfied": ((B,), torch.int32), "step": ((B,), torch.int32), "done": ((B, d.A), torch.uint8),
            "clauses": ((B, d.m, d.k), torch.int32), "agent_clause_masks": ((B, d.A, d.m), torch.int32),
            "agent_neighbor_masks": ((B, d.A, d.n), torch.int32), "literal_to_agent_idx": ((B, d.m, d.k), torch.int32),
            "problem_idx": ((B,), torch.int32),
        }
        shape, dtype = shapes[name]
        out = torch.empty(shape, dtype=dtype, device=dev)
        ptrs = [_ptr(out) if leaf == name else None for leaf in self._EXPORT_ORDER]
        _lib.check(env._lib.msat_export_state(
            self.bank.plan.handle, _ptr(self.bank.data), self.bank.num_problems, _ptr(self.packed), B, *ptrs,
            _stream_ptr(dev)), "msat_export_state")
        if name in ("clauses_satisfied_status", "done"):
            out = out.bool()
        self._cache[name] = out


def _make_leaf_property(name):
    return property(lambda self: self._leaf(name))


for _name in SATState._LEAVES:
    setattr(SATState, _name, _make_leaf_property(_name))


class SATEnv:
    """Batched multi-agent SAT environment (drop-in for env:28-411)."""

    def __init__(self, num_vars, num_clauses, max_steps: int, vars_per_agent: Optional[int] = None,
                 action_mode: int = 0, r_clause: float = 0.02, r_sat: float = 1.0, gamma: float = 0.99,
                 *, device: Union[str, torch.device, None] = None, verbose: bool = True,
                 group_threads: int = 0, reward_mode: str = "sparse", clause_update: str = "full",
                 obs_dtype: Union[str, torch.dtype] = torch.int32):
        self._lib = _lib.load()
        # int32 is what the reference declares (env:390-396) and the default; int8 carries the same -1 / 0 / 1
        # values in a quarter of the bytes for consumers that cast the observations anyway (MSAT_OBS_INT8)
        obs_dtype = {"int32": torch.int32, "int8": torch.int8}.get(obs_dtype, obs_dtype)
        if obs_dtype not in (torch.int32, torch.int8):
            raise ValueError("obs_dtype must be torch.int32 (the reference's) or torch.int8")
        self.obs_dtype = obs_dtype
        self.num_vars = int(num_vars)
        self.num_clauses = int(num_clauses)
        self.agent_groups = create_agent_groups(self.num_vars, vars_per_agent, verbose=verbose)
        self.agents = list(self.agent_groups.keys())
        self.num_agents = len(self.agents)
        self.agent_to_idx = {a: i for i, a in enumerate(self.agents)}
        # stored but unused by the reference's active reward (env:40-42,183-198); reward_mode="shaped" selects
        # the alternative team reward the reference keeps commented out (env:201-223), which does use them
        self.r_clause, self.r_sat, self.gamma = r_clause, r_sat, gamma
        if reward_mode not in ("sparse", "shaped"):
            raise ValueError("reward_mode must be 'sparse' or 'shaped'")
        self.reward_mode = reward_mode
        # "incremental": launches without observations update per-clause true-literal counts from the var ->
        # clause occurrence lists of the flipped variables instead of re-evaluating every clause (same results)
        if clause_update not in ("full", "incremental"):
            raise ValueError("clause_update must be 'full' or 'incremental'")
        self.clause_update = clause_update
        self.action_mode = int(action_mode)
        self.max_steps = int(max_steps)
        self.max_vars_per_agent = max(len(v) for v in self.agent_groups.values())
        self._group_threads = int(group_threads)
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else torch.device("cpu")
        self.device = torch.device(device)

        A, V = self.num_agents, self.max_vars_per_agent
        av = np.full((A, V), -1, dtype=np.int32)                              # env:61
        am = np.zeros((A, V), dtype=bool)                                     # env:62
        v2a = np.full((self.num_vars,), -1, dtype=np.int32)                   # env:92-97
        for i, a in enumerate(self.agents):
            vs = self.agent_groups[a]
            av[i, :len(vs)] = vs
            am[i, :len(vs)] = True
            v2a[vs] = i
        self.agent_vars = torch.from_numpy(av).to(self.device)
        self.action_mask = torch.from_numpy(am).to(self.device)
        self.variable_to_agent_idx = torch.from_numpy(v2a).to(self.device)

        self.action_spaces = {}
        for a in self.agents:                                                 # env:68-79
            if self.action_mode == 0:
                self.action_spaces[a] = spaces.Discrete(V + 1, dtype=torch.int32)
            else:
                self.action_spaces[a] = spaces.MultiDiscrete([2] * V)
        self.obs_dim = self._calculate_obs_dim()
        self.observation_spaces = {a: spaces.Box(-1, 1, (self.obs_dim,)) for a in self.agents}   # env:84
        self._plans: Dict[int, _Plan] = {}

    # ------------------------------------------------------------------ helpers
    def _calculate_obs_dim(self) -> int:                                      # env:340-343
        return self.num_vars + self.num_clauses + self.num_vars

    def _require_cuda(self) -> torch.device:
        if self.device.type != "cuda" or not torch.cuda.is_available():
            raise RuntimeError("marl_sat_b200.SATEnv needs a CUDA device: there is no CPU fallback")
        return self.device

    def _plan_for(self, k: int) -> _Plan:
        if k not in self._plans:
            reward = (1, float(self.gamma), float(self.r_clause), float(self.r_sat)) if self.reward_mode == "shaped" else None
            self._plans[k] = _Plan(self.num_vars, self.num_clauses, k, self.num_agents, self.action_mode,
                                   self.max_steps, self._group_threads, reward,
                                   incremental=self.clause_update == "incremental",
                                   obs_int8=self.obs_dtype == torch.int8)
        return self._plans[k]

    def count_resets(self, k: int, counter: Optional[torch.Tensor]) -> None:
        """Diagnostics: route the auto-reset count of every step launch on formulas of width ``k`` into
        ``counter`` (a zeroed int64[1] device tensor), or switch it off with ``None``."""
        _lib.check(self._lib.msat_plan_set_reset_counter(self._plan_for(k).handle, _ptr(counter)),
                   "msat_plan_set_reset_counter")

    def make_bank(self, clauses: ArrayLike, validate: bool = True) -> FormulaBank:
        return FormulaBank(self, clauses, validate=validate)

    @property
    def name(self) -> str:                                                    # env:401-404
        return "SATEnv"

    def action_space(self, agent: str):                                       # env:406-407
        return self.action_spaces[agent]

    def observation_space(self, agent: str):                                  # env:409-411
        return self.observation_spaces[agent]

    # ------------------------------------------------------------------ reset
    def reset(self, problem_clauses: ArrayLike, key: ArrayLike) -> Tuple[Dict[str, torch.Tensor], SATState]:
        """``reset(problem_clauses[m,k], key[2])`` (env:158-181) or its vmapped form
        ``reset(problem_clauses[B,m,k], keys[B,2])`` (runner:137)."""
        dev = self._require_cuda()
        cl = problem_clauses if isinstance(problem_clauses, torch.Tensor) else torch.as_tensor(np.asarray(problem_clauses))
        batched = cl.dim() == 3
        if not batched:
            cl = cl[None]
        bank = FormulaBank(self, cl)
        B = bank.num_problems
        keys = as_u32_tensor(key, dev).reshape(-1, 2)
        if keys.shape[0] != B:
            raise ValueError(f"need one PRNG key per env: got {tuple(keys.shape)} for {B} formulas")
        idx = torch.arange(B, dtype=torch.int32, device=dev)
        obs, state = self.reset_from_bank(bank, idx, keys)
        state.batched = batched
        return self._obs_dict(obs, batched), state

    def reset_from_bank(self, bank: FormulaBank, problem_idx: torch.Tensor, keys: torch.Tensor,
                        state_out: Optional[torch.Tensor] = None, obs_out: Optional[torch.Tensor] = None,
                        want_obs: bool = True, validate_indices: bool = False) -> Tuple[Optional[torch.Tensor], SATState]:
        """Batched reset on formulas already resident in a bank: obs ``int32[B,A,D]`` + state.
        The kernels clamp a problem index into ``[0, P)``; ``validate_indices=True`` checks the range on the
        host first (one device->host sync) and raises instead."""
        dev = self._require_cuda()
        d = bank.plan.dims
        B = int(problem_idx.shape[0])
        problem_idx = problem_idx.to(device=dev, dtype=torch.int32).contiguous()
        if validate_indices and B:
            lo, hi = int(problem_idx.min()), int(problem_idx.max())
            if lo < 0 or hi >= bank.num_problems:
                raise IndexError(f"problem_idx out of range [0, {bank.num_problems}): min {lo}, max {hi}")
        keys = as_u32_tensor(keys, dev)
        packed = state_out if state_out is not None else torch.empty((B, d.state_words), dtype=torch.int32, device=dev)
        obs = obs_out
        if obs is None and want_obs:
            obs = obs_empty((B, d.A, d.D), self.obs_dtype, dev)
        _lib.check(self._lib.msat_reset(bank.plan.handle, _ptr(bank.data), bank.num_problems, _ptr(problem_idx),
                                        _ptr(keys), _ptr(packed), _ptr(obs), B, _stream_ptr(dev)), "msat_reset")
        return obs, SATState(self, bank, packed, True)

    # ------------------------------------------------------------------ state import
    def reset_with_assignment(self, problem_clauses: ArrayLike, variable_assignments: ArrayLike,
                              step: Optional[ArrayLike] = None,
                              done: Optional[ArrayLike] = None) -> Tuple[Dict[str, torch.Tensor], SATState]:
        """Counterpart of ``reset(problem_clauses, key)`` (env:158-181) that starts from a given assignment instead
        of a random one: ``(problem_clauses[m,k], variable_assignments[n])`` or the batched ``[B,m,k]`` / ``[B,n]``.
        ``step`` / ``done`` (default 0 / False) as in ``import_state``."""
        self._require_cuda()
        cl = problem_clauses if isinstance(problem_clauses, torch.Tensor) else torch.as_tensor(np.asarray(problem_clauses))
        batched = cl.dim() == 3
        va = torch.as_tensor(np.asarray(variable_assignments)) if not isinstance(variable_assignments, torch.Tensor) \
            else variable_assignments
        if not batched:
            cl, va = cl[None], va.reshape(1, -1)
            if step is not None:
                step = torch.as_tensor(step).reshape(1)
            if done is not None:
                done = torch.as_tensor(done)
                done = done.reshape(1) if done.numel() == 1 else done.reshape(1, -1)
        bank = FormulaBank(self, cl)
        idx = torch.arange(bank.num_problems, dtype=torch.int32, device=self.device)
        obs, state = self.import_state(bank, idx, va, step, done)
        state.batched = batched
        return self._obs_dict(obs, batched), state

    def import_state(self, bank: FormulaBank, problem_idx: ArrayLike, variable_assignments: ArrayLike,
                     step: Optional[ArrayLike] = None, done: Optional[ArrayLike] = None, *,
                     state_out: Optional[torch.Tensor] = None, obs_out: Optional[torch.Tensor] = None,
                     want_obs: bool = True, validate: bool = True) -> Tuple[Optional[torch.Tensor], SATState]:
        """Inverse of the ``SATState`` export (``msat_import_state``): packed states of formulas resident in
        ``bank`` built from reference-shaped leaves (env:13-24), and their observations ``[B,A,D]``.  Mirrors
        ``reset_from_bank``.
          variable_assignments  int32 / uint8 / bool ``[B, n]``, values 0 / 1
          step                  int ``[B]``, default 0; stored as given, also at or past ``max_steps``
          done                  ``[B]`` or the reference's per-agent ``[B, A]``, default False
        Clause status, ``num_unsatisfied`` (and an incremental plan's per-clause counts) are recomputed on the
        device.  ``validate=True`` checks on the host that assignments are 0 / 1, ``step >= 0``, problem indices
        lie in ``[0, P)`` and ``[B, A]`` done rows are uniform (one device->host sync; ValueError / IndexError).
        ``validate=False`` enqueues only and can be captured in a CUDA graph: the kernel then clamps problem indices
        into ``[0, P)``, reads a nonzero assignment as 1 and takes agent 0's done flag."""
        dev = self._require_cuda()
        d = bank.plan.dims
        idx = torch.as_tensor(problem_idx)
        if idx.dim() != 1:
            raise ValueError(f"problem_idx must be [B], got {tuple(idx.shape)}")
        B = int(idx.shape[0])
        idx = idx.to(device=dev, dtype=torch.int32).contiguous()
        va = torch.as_tensor(variable_assignments)
        if va.dtype not in (torch.int32, torch.uint8, torch.bool):
            raise ValueError(f"variable_assignments must be int32, uint8 or bool, got {va.dtype}")
        if tuple(va.shape) != (B, d.n):
            raise ValueError(f"variable_assignments must be [{B}, {d.n}], got {tuple(va.shape)}")
        va = va.to(device=dev, dtype=torch.int32).contiguous()
        st = None
        if step is not None:
            st = torch.as_tensor(step)
            if tuple(st.shape) != (B,):
                raise ValueError(f"step must be [{B}], got {tuple(st.shape)}")
            st = st.to(device=dev, dtype=torch.int32).contiguous()
        dn = dn_rows = None
        if done is not None:
            dn_rows = torch.as_tensor(done).to(device=dev)
            if tuple(dn_rows.shape) not in ((B,), (B, d.A)):
                raise ValueError(f"done must be [{B}] or [{B}, {d.A}], got {tuple(dn_rows.shape)}")
            dn = ((dn_rows[:, 0] if dn_rows.dim() == 2 else dn_rows) != 0).to(torch.uint8).contiguous()
        if state_out is not None and tuple(state_out.shape) != (B, d.state_words):
            raise ValueError(f"state_out must be [{B}, {d.state_words}], got {tuple(state_out.shape)}")
        if validate and B:
            zero = torch.zeros((), dtype=torch.int64, device=dev)
            nz = dn_rows != 0 if dn_rows is not None and dn_rows.dim() == 2 else None
            lo, hi, bad_assign, min_step, mixed_done = torch.stack([
                idx.min().long(), idx.max().long(), ((va != 0) & (va != 1)).any().long(),
                st.min().long() if st is not None else zero,
                (nz.any(1) != nz.all(1)).any().long() if nz is not None else zero]).tolist()
            if lo < 0 or hi >= bank.num_problems:
                raise IndexError(f"problem_idx out of range [0, {bank.num_problems}): min {lo}, max {hi}")
            if bad_assign:
                raise ValueError("variable_assignments must hold 0 / 1 values only")
            if min_step < 0:
                raise ValueError(f"step must be >= 0, got min {min_step}")
            if mixed_done:
                raise ValueError("done [B, A]: every agent of an env must carry the same flag (env:260)")
        packed = state_out if state_out is not None else torch.empty((B, d.state_words), dtype=torch.int32, device=dev)
        obs = obs_out
        if obs is None and want_obs:
            obs = obs_empty((B, d.A, d.D), self.obs_dtype, dev)
        _lib.check(self._lib.msat_import_state(bank.plan.handle, _ptr(bank.data), bank.num_problems, _ptr(idx),
                                               _ptr(va), _ptr(st), _ptr(dn), _ptr(packed), _ptr(obs), B,
                                               _stream_ptr(dev)), "msat_import_state")
        return obs, SATState(self, bank, packed, True)

    # ------------------------------------------------------------------ step
    def _actions_tensor(self, actions, B: int, dev) -> torch.Tensor:
        if isinstance(actions, dict):                                         # learner:131
            parts = [torch.as_tensor(actions[a]).to(dev) for a in self.agents]
            actions = torch.stack(parts, dim=-1) if self.action_mode == 0 else torch.stack(parts, dim=-2)
        act = torch.as_tensor(actions).to(device=dev, dtype=torch.int32)
        shape = (B, self.num_agents) if self.action_mode == 0 else (B, self.num_agents, self.max_vars_per_agent)
        if act.numel() != math.prod(shape):
            raise ValueError(f"actions must have shape {shape} (or unbatched), got {tuple(act.shape)}")
        return act.reshape(shape).contiguous()

    def step_env(self, key, state: SATState, actions_array):
        """``step_env(key, state, actions_array)`` (env:225-284): returns
        ``(obs, next_state, rewards, dones, infos)``.  ``key`` is unused, as in the reference."""
        del key
        dev = self._require_cuda()
        d = state.bank.plan.dims
        B = state.num_envs
        act = self._actions_tensor(actions_array, B, dev)
        out = self.alloc_step_outputs(B, d)
        new_packed = torch.empty_like(state.packed)
        self.step_into(state.bank, state.packed, new_packed, act, out)
        nxt = SATState(self, state.bank, new_packed, state.batched)
        b = state.batched
        sq = (lambda t: t) if b else (lambda t: t[0])
        rewards = {a: sq(out["reward"][:, i]) for i, a in enumerate(self.agents)}        # env:196
        done_b = out["done"].bool()
        dones = {a: sq(done_b[:, i]) for i, a in enumerate(self.agents)}                 # env:260
        dones["__all__"] = sq(done_b[:, self.num_agents])                                # env:261
        infos = {"solved": sq(out["solved"].bool()), "num_unsatisfied": sq(out["num_unsatisfied"]),
                 "episode_step": sq(out["episode_step"])}                                # env:278-282
        if out["newly_satisfied"] is not None:
            infos["newly_satisfied"] = sq(out["newly_satisfied"])                         # env:211 (shaped reward only)
        return self._obs_dict(out["obs"], b), nxt, rewards, dones, infos

    def step(self, key, state, actions):
        """jaxmarl's auto-resetting ``MultiAgentEnv.step`` calls ``self.reset(key)``; the reference
        overrides ``reset(problem_clauses, key)`` so that path raises there too.  Use ``step_env``
        (or ``VecSATEnv`` for the rollout auto-reset of learner:422-464)."""
        raise TypeError("SATEnv.step() is unusable in the reference (reset needs problem_clauses); "
                        "call step_env(key, state, actions_array) or use marl_sat_b200.VecSATEnv")

    def alloc_step_outputs(self, B: int, d=None, want_obs: bool = True, compact: bool = False,
                           pinned_host: bool = False) -> Dict[str, torch.Tensor]:
        """Output buffers of one step.  ``compact=True`` keeps one reward / done column per env (the shared
        team reward and ``done["__all__"]``) instead of one per agent.  reward, num_unsatisfied,
        episode_step, done and solved are views of ONE block (in that order, 4-byte fields first) so that a
        host mirror allocated with ``pinned_host=True`` receives them in a single transfer."""
        A, D = self.num_agents, self.obs_dim
        rc, dc = (1, 1) if compact else (A, A + 1)
        if pinned_host:
            block = torch.empty(B * (4 * rc + 8 + dc + 1), dtype=torch.uint8, pin_memory=True)
            obs = None
        else:
            dev = self._require_cuda()
            block = torch.empty(B * (4 * rc + 8 + dc + 1), dtype=torch.uint8, device=dev)
            obs = obs_empty((B, A, D), self.obs_dtype, dev) if want_obs else None
        o0, o1, o2, o3 = 4 * rc * B, 4 * rc * B + 4 * B, 4 * rc * B + 8 * B, 4 * rc * B + 8 * B + dc * B
        newly = None
        if self.reward_mode == "shaped":
            newly = (torch.empty(B, dtype=torch.int32, pin_memory=True) if pinned_host
                     else torch.empty(B, dtype=torch.int32, device=self._require_cuda()))
        return {
            "obs": obs,
            "newly_satisfied": newly,
            "reward": block[:o0].view(torch.float32).view(B, rc),
            "num_unsatisfied": block[o0:o1].view(torch.int32),
            "episode_step": block[o1:o2].view(torch.int32),
            "done": block[o2:o3].view(B, dc),
            "solved": block[o3:],
            "_block": block,
        }

    def step_into(self, bank: FormulaBank, state_in: torch.Tensor, state_out: torch.Tensor, actions: torch.Tensor,
                  out: Dict[str, Optional[torch.Tensor]], auto_reset: bool = False,
                  new_problem_idx: Optional[torch.Tensor] = None, reset_keys: Optional[torch.Tensor] = None) -> None:
        """Thin call of ``msat_step`` on preallocated device tensors (enqueue only, graph-capturable)."""
        B = int(state_in.shape[0])
        done, reward = out.get("done"), out.get("reward")
        _lib.check(self._lib.msat_step(
            bank.plan.handle, _ptr(bank.data), bank.num_problems, _ptr(state_in), _ptr(state_out), _ptr(actions),
            1 if auto_reset else 0, _ptr(new_problem_idx), _ptr(reset_keys),
            _ptr(out.get("obs")), _ptr(reward), int(reward.shape[-1]) if reward is not None else 0,
            _ptr(done), int(done.shape[-1]) if done is not None else 0, _ptr(out.get("solved")),
            _ptr(out.get("num_unsatisfied")), _ptr(out.get("episode_step")), _ptr(out.get("newly_satisfied")), B,
            _stream_ptr(state_in.device)), "msat_step")

    # ------------------------------------------------------------------ observations
    def get_obs_array(self, state: SATState) -> torch.Tensor:
        dev = self._require_cuda()
        d = state.bank.plan.dims
        B = state.num_envs
        obs = obs_empty((B, d.A, d.D), self.obs_dtype, dev)
        _lib.check(self._lib.msat_get_obs(state.bank.plan.handle, _ptr(state.bank.data), state.bank.num_problems,
                                          _ptr(state.packed), _ptr(obs), B, _stream_ptr(dev)), "msat_get_obs")
        return obs

    def get_obs(self, state: SATState) -> Dict[str, torch.Tensor]:           # env:345-398
        return self._obs_dict(self.get_obs_array(state), state.batched)

    def _obs_dict(self, obs: torch.Tensor, batched: bool) -> Dict[str, torch.Tensor]:
        """Per-agent views of the single ``[B, A, D]`` buffer (the reference returns a dict keyed by agent)."""
        if batched:
            return {a: obs[:, i] for i, a in enumerate(self.agents)}
        return {a: obs[0, i] for i, a in enumerate(self.agents)}
