"""Rollout-side host logic: the per-step RNG chain, fused auto-reset stepping and the rollout buffer.

Mirrors the env half of ``_env_step`` in the reference learner
(``/root/reference/src/learners/mappo_gnn_sat_learner.py:383-480``, cited as learner:LINE) and the
initial reset of the runner (``src/runners/mappo_runner.py:289-295``, runner:LINE):

    rng, act_key  = split(rng)                      learner:397   (policy sampling key)
    rng, step_key = split(rng)                      learner:416   (unused by SATEnv)
    step all envs                                   learner:418
    rng, prob_key, reset_key = split(rng, 3)        learner:426
    new_problem_indices = randint(prob_key, B, P)   learner:430
    reset_keys = split(reset_key, B)                learner:434
    reset finished envs on their new formula        learner:435-464  (the reference resets *every*
                                                    env and selects with where(done); the kernel
                                                    resets only finished envs -- same result)

Environments shard across ranks as contiguous blocks of the global batch with no data-path
collective; the per-env keys are derived from *global* env indices so that any sharding yields the
values of the single-device run (SURVEY.md section 8e).
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Tuple

import numpy as np
import torch

from . import _lib
from .curriculum import StartTable, problem_stats, problem_weights, start_table
from .env import ArrayLike, FormulaBank, SATEnv, SATState, _ptr, _stream_ptr, as_u32_tensor, obs_empty
from .sampling import sample_actions


def prng_key(seed: int):
    """``jax.random.PRNGKey(seed)`` as a legacy uint32[2] key: ``[seed >> 32, seed & 0xFFFFFFFF]``."""
    import numpy as np
    return np.array([(seed >> 32) & 0xFFFFFFFF, seed & 0xFFFFFFFF], dtype=np.uint32)


def shard_range(num_envs_global: int, world_size: int, rank: int):
    """Contiguous block ``[offset, offset + count)`` of the global env batch owned by ``rank``."""
    base, rem = divmod(num_envs_global, world_size)
    count = base + (1 if rank < rem else 0)
    offset = rank * base + min(rank, rem)
    return offset, count


class RolloutKeys:
    """Device-resident ``rng`` of the rollout carry and the per-step chain derived from it.

    Two 10-word buffers are used alternately so that the fused step kernel can read the current rng
    from one while it writes the advanced chain ``{rng', act, step, prob, reset}`` into the other."""

    def __init__(self, key, device: torch.device):
        self.device = device
        self._lib = _lib.load()
        self._bufs = torch.zeros((2, 10), dtype=torch.int32, device=device)
        self._cur = 0
        self._bufs[0, :2] = as_u32_tensor(key, device).reshape(2)
        self._buf_ptrs = (self._bufs[0].data_ptr(), self._bufs[1].data_ptr())   # _bufs is only ever updated in place

    @property
    def chain(self) -> torch.Tensor:
        """uint32[10] (as int32 bits): rng, act_key, step_key, prob_key, reset_key of the latest step."""
        return self._bufs[self._cur]

    @property
    def next_chain(self) -> torch.Tensor:
        return self._bufs[1 - self._cur]

    def flip(self) -> None:
        self._cur = 1 - self._cur

    def take_launch_ptrs(self) -> Tuple[int, int]:
        """Device pointers of ``(chain, next_chain)`` -- the ``rng_in`` / ``chain_out`` of a launch that advances the
        chain -- and ``flip``: the launch's chain becomes current.  ``flip`` again if the launch fails."""
        cur = self._cur
        self._cur = 1 - cur
        return self._buf_ptrs[cur], self._buf_ptrs[1 - cur]

    @property
    def rng(self) -> torch.Tensor:
        return self.chain[0:2]

    @property
    def act_key(self) -> torch.Tensor:
        return self.chain[2:4]

    @property
    def step_key(self) -> torch.Tensor:
        return self.chain[4:6]

    @property
    def prob_key(self) -> torch.Tensor:
        return self.chain[6:8]

    @property
    def reset_key(self) -> torch.Tensor:
        return self.chain[8:10]

    def advance(self) -> None:
        """One rollout step of the chain (learner:397,416,426), enqueue only."""
        _lib.check(self._lib.msat_rng_chain(_ptr(self.chain), _ptr(self.next_chain), _stream_ptr(self.device)),
                   "msat_rng_chain")
        self.flip()


# Per-call arguments of a bound rollout launch: placeholders in the argument list that _BoundCall fills in on every call
# (ctypes rejects one left unfilled).
_ACTIONS, _RNG_IN, _CHAIN_OUT, _STREAM = object(), object(), object(), object()


class _BoundCall:
    """A rollout entry point with its argument list built once (``VecSATEnv._bind``).  A call fills the per-call
    slots -- the action pointers it is given, the rng buffers of ``keys`` and the device's current stream (a graph
    capture runs on a side stream) -- launches and advances ``keys``, or raises on an error code."""

    def __init__(self, fn, name: str, args: list, keys: RolloutKeys, device: torch.device):
        self.fn, self.name, self.args, self.keys, self.device = fn, name, args, keys, device
        first = args.index(_ACTIONS)
        self.actions = slice(first, first + args.count(_ACTIONS))
        assert all(a is _ACTIONS for a in args[self.actions]), f"{name}: the action pointers must be adjacent"
        self.rng_in, self.chain_out, self.stream = args.index(_RNG_IN), args.index(_CHAIN_OUT), args.index(_STREAM)

    def __call__(self, *action_ptrs: int) -> None:
        args = self.args
        args[self.actions] = action_ptrs
        args[self.rng_in], args[self.chain_out] = self.keys.take_launch_ptrs()
        args[self.stream] = torch.cuda.current_stream(self.device).cuda_stream
        rc = self.fn(*args)
        if rc != 0:
            self.keys.flip()
            _lib.check(rc, self.name)


def derive_env_keys(prob_key: Optional[torch.Tensor], reset_key: Optional[torch.Tensor], num_envs_global: int,
                    env_offset: int, num_envs_local: int, num_problems: int,
                    problem_idx: Optional[torch.Tensor], reset_keys: Optional[torch.Tensor],
                    cum_weights: Optional[torch.Tensor] = None) -> None:
    """``randint(prob_key, (Bg,), 0, P)`` and ``split(reset_key, Bg)`` restricted to a shard.  With ``cum_weights``
    (int64 ``[P]`` device tensor, inclusive prefix sums of ``curriculum.problem_weights``) the problem indices come
    from the weighted draw of ``msat_env_keys_weighted`` instead; the reset keys are the same."""
    lib = _lib.load()
    dev = (problem_idx if problem_idx is not None else reset_keys).device
    if cum_weights is None:
        _lib.check(lib.msat_env_keys(_ptr(prob_key), _ptr(reset_key), num_envs_global, env_offset, num_envs_local,
                                     num_problems, _ptr(problem_idx), _ptr(reset_keys), _stream_ptr(dev)),
                   "msat_env_keys")
        return
    if cum_weights.dtype != torch.int64 or tuple(cum_weights.shape) != (num_problems,) or cum_weights.device != dev:
        raise ValueError(f"cum_weights must be an int64 [{num_problems}] tensor on {dev}")
    _lib.check(lib.msat_env_keys_weighted(_ptr(prob_key), _ptr(reset_key), num_envs_global, env_offset,
                                          num_envs_local, _ptr(cum_weights.contiguous()), num_problems,
                                          _ptr(problem_idx), _ptr(reset_keys), _stream_ptr(dev)),
               "msat_env_keys_weighted")


class VecSATEnv:
    """B parallel SATEnv episodes with the reference's auto-reset and RNG chain fused on device.

    One instance per process/GPU; ``world_size``/``rank`` select the shard of the global batch.
    All per-step work is enqueue-only on the current stream (no host sync, graph-capturable).
    """

    def __init__(self, env: SATEnv, problems: FormulaBank | torch.Tensor, num_envs: int, key,
                 world_size: int = 1, rank: int = 0, emit_obs: bool = True, fused_keys: bool = True,
                 compact_outputs: bool = False, gnn_outputs: bool = False):
        self.env = env
        self.fused_keys = fused_keys
        dev = env._require_cuda()
        self.bank = problems if isinstance(problems, FormulaBank) else env.make_bank(problems)
        self.num_envs_global = int(num_envs)
        self.env_offset, self.num_envs = shard_range(self.num_envs_global, world_size, rank)
        self.keys = RolloutKeys(key, dev)
        d = self.bank.plan.dims
        B = self.num_envs
        self.state = torch.empty((B, d.state_words), dtype=torch.int32, device=dev)
        self.new_problem_idx = torch.empty((B,), dtype=torch.int32, device=dev)
        self.reset_keys = torch.empty((B, 2), dtype=torch.int32, device=dev)
        self.out = env.alloc_step_outputs(B, d, want_obs=emit_obs, compact=compact_outputs)
        self._split_tmp = torch.empty(4, dtype=torch.int32, device=dev)
        # GNN-style consumers: the step emits assignment / clause features instead of local observations
        self.gnn_outputs = gnn_outputs
        if gnn_outputs:
            self.out["gnn_assignment"] = torch.empty((B, d.n), dtype=torch.int32, device=dev)
            self.out["gnn_clause_features"] = torch.empty((B, d.m, 3), dtype=torch.float32, device=dev)
        self._weights: Optional[torch.Tensor] = None        # quantised problem weights (host), None = uniform draw
        self._cum_weights: Optional[torch.Tensor] = None    # their inclusive prefix sums on the device
        self._start: Optional[StartTable] = None             # start-state tables (host), None = random starts
        self._start_dev: Optional[Dict[str, torch.Tensor]] = None   # their device copies, allocated once
        # bindings (_bind) cached with the buffers they were built over: at small per-GPU batches the ~80 µs kernel
        # is short enough for per-call Python work to matter
        self._fast_args = None   # step() on self.out: (binding, self.out["obs"])
        self._host_args = None   # step_host: (binding, host["reward"], self.out["obs"])

    # ------------------------------------------------------------------ weighted problem draw
    @property
    def problem_weights(self) -> Optional[torch.Tensor]:
        """The quantised weights of ``set_problem_weights`` (int64 ``[P]``, host), or None for the uniform draw."""
        return self._weights

    def set_problem_weights(self, weights: Optional[ArrayLike]) -> None:
        """Draw the problems of ``reset`` and of every auto-reset with probability proportional to ``weights``
        (``[P]``, non-negative, not all zero; quantised by ``curriculum.problem_weights``) instead of uniformly.
        ``None`` restores the uniform draw and the fused one-launch step.  Every rank must pass the same weights:
        each env's draw depends only on the rng, its global index and the weights, which keeps sharded runs equal to
        the single-device run.  The weights are validated on the host and copied into a device buffer that this env
        allocates once, so changing them between replays of a captured CUDA graph needs no re-capture.  While
        weights are set, ``step`` runs ``msat_rng_chain`` -> ``msat_env_keys_weighted`` -> ``msat_step`` (three
        launches), and ``steps``, ``step_host`` and ``step_host_async`` raise ``ValueError``."""
        if weights is None:
            self._weights = None
            return
        self._install_weights(problem_weights(weights, self.bank.num_problems))

    def _install_weights(self, q: torch.Tensor) -> None:
        if self._cum_weights is None:
            self._cum_weights = torch.empty((self.bank.num_problems,), dtype=torch.int64, device=self.state.device)
        self._cum_weights.copy_(torch.cumsum(q, 0))
        self._weights = q

    def _require_plain_resets(self, what: str) -> None:
        """Refuse a fused entry point that resets envs itself while problem weights or start states are set."""
        if self._weights is not None:
            raise ValueError(f"{what} draws problem indices inside its fused kernel and cannot apply problem weights; "
                             f"use step(), or set_problem_weights(None) first")
        if self._start is not None:
            raise ValueError(f"{what} resets envs inside its fused kernel and cannot apply start states; "
                             f"use step(), or set_start_states(None) first")

    # ------------------------------------------------------------------ start states (reverse curriculum)
    @property
    def start_states(self) -> Optional[StartTable]:
        """The tables of ``set_start_states`` (``curriculum.StartTable``, host), or None for random starts."""
        return self._start

    def set_start_states(self, assignments: Optional[ArrayLike], flip_prob=0.0,
                         has_start: Optional[ArrayLike] = None) -> None:
        """Start every reset episode of a problem with a start at that problem's stored assignment, each bit flipped
        with probability ``flip_prob`` (a scalar or ``[P]``), instead of at the random draw (a reverse curriculum).
        ``assignments`` ``[P, n]`` (nonzero = 1; e.g. WalkSAT solutions), ``has_start`` ``[P]`` (default every
        problem); the tables are built by ``curriculum.start_table``.  While starts are set, ``reset`` and every
        ``step`` end with ``msat_apply_start_states`` on that call's reset key, so only envs that just restarted are
        rewritten, and each one's start depends only on the rng, its global index and the tables: sharded runs equal
        the single-device run.  The device tables are allocated once and updated in place, so a captured CUDA graph
        picks up new values without re-capture.  ``steps``, ``step_host`` and ``step_host_async`` raise
        ``ValueError`` while starts are set.  ``None`` removes the extra launch."""
        if assignments is None:
            self._start = None
            return
        d = self.bank.plan.dims
        shape = tuple(assignments.shape) if hasattr(assignments, "shape") else np.shape(assignments)
        if tuple(shape) != (self.bank.num_problems, d.n):
            raise ValueError(f"start assignments must be [{self.bank.num_problems}, {d.n}], got {tuple(shape)}")
        self._install_starts(start_table(assignments, flip_prob, has_start))

    def _install_starts(self, table: StartTable) -> None:
        dev = self.state.device
        if self._start_dev is None:
            P, aw = table.words.shape
            self._start_dev = {"words": torch.empty((P, aw), dtype=torch.int32, device=dev),
                               "flip_thr": torch.empty((P,), dtype=torch.int32, device=dev),
                               "has_start": torch.empty((P,), dtype=torch.uint8, device=dev)}
        t = self._start_dev
        t["words"].copy_(table.words)
        t["flip_thr"].copy_(table.flip_thr.to(torch.int64).bitwise_and(0xFFFFFFFF).to(torch.int32))  # uint32 bits
        t["has_start"].copy_(table.has_start)
        self._start = StartTable(table.words.clone(), table.flip_thr.clone(), table.has_start.clone())

    def _apply_starts(self, reset_key: torch.Tensor, obs: Optional[torch.Tensor],
                      gnn: Optional[Dict[str, torch.Tensor]] = None) -> None:
        t = self._start_dev
        _lib.check(self.env._lib.msat_apply_start_states(
            self.bank.plan.handle, _ptr(self.bank.data), self.bank.num_problems, _ptr(self.state), _ptr(reset_key),
            self.num_envs_global, self.env_offset, _ptr(t["words"]), _ptr(t["flip_thr"]), _ptr(t["has_start"]),
            _ptr(obs), _ptr(gnn["gnn_assignment"]) if gnn else None, _ptr(gnn["gnn_clause_features"]) if gnn else None,
            self.num_envs, _stream_ptr(self.state.device)), "msat_apply_start_states")

    # runner:289-295 -- key,_rng = split(key); idx = randint(_rng,...); reset_keys = split(_rng, B)
    def reset(self) -> Optional[torch.Tensor]:
        lib, dev = self.env._lib, self.state.device
        _lib.check(lib.msat_rng_split2(_ptr(self.keys.chain), _ptr(self._split_tmp), _stream_ptr(dev)), "msat_rng_split2")
        self.keys.chain[0:2].copy_(self._split_tmp[0:2])     # key
        rng = self._split_tmp[2:4]                           # _rng, used for both draws (runner:291,294)
        derive_env_keys(rng, rng, self.num_envs_global, self.env_offset, self.num_envs, self.bank.num_problems,
                        self.new_problem_idx, self.reset_keys, None if self._weights is None else self._cum_weights)
        obs, _ = self.env.reset_from_bank(self.bank, self.new_problem_idx, self.reset_keys, state_out=self.state,
                                          obs_out=self.out["obs"], want_obs=self.out["obs"] is not None)
        if self._start is not None:
            self._apply_starts(rng, self.out["obs"])
        return obs

    def step(self, actions: torch.Tensor, out: Optional[Dict[str, torch.Tensor]] = None) -> Dict[str, torch.Tensor]:
        """One rollout step (learner:397-464) for this shard.  ``actions`` int32 ``[B, A]`` (mode 0) or
        ``[B, A, V]`` (mode 1) on the device.  Returns the output dict (obs of the state to continue
        from; reward/done/info are the pre-reset values, learner:467-478).  With ``gnn_outputs`` the step emits the
        dynamic GNN input into ``self.out`` instead of local observations (``msat_rollout_step_gnn``; combine with
        ``features.static_graph(bank)`` for the full ``GNNInput``).  While start states are set, the envs that
        restarted are then moved to their starts (``msat_apply_start_states`` with this step's reset key)."""
        res = self._step(actions, out)
        if self._start is not None:
            if self.gnn_outputs:
                self._apply_starts(self.keys.reset_key, None, self.out)
            else:
                self._apply_starts(self.keys.reset_key, res.get("obs"))
        return res

    def _step(self, actions: torch.Tensor, out: Optional[Dict[str, torch.Tensor]]) -> Dict[str, torch.Tensor]:
        weighted = self._weights is not None
        if not weighted and (self.gnn_outputs or self.fused_keys):
            # one launch: rng chain + per-env key derivation + step + auto-reset; the GNN-input step ignores ``out``
            if out is not None and not self.gnn_outputs:
                self._bind("msat_rollout_step", out)(actions.data_ptr())
                return out
            call, obs = self._fast_args or (None, None)
            if call is None or obs is not self.out["obs"]:
                call = self._bind("msat_rollout_step_gnn" if self.gnn_outputs else "msat_rollout_step", self.out)
                self._fast_args = (call, self.out["obs"])
            call(actions.data_ptr())
            return self.out
        out = self.out if out is None or self.gnn_outputs else out
        # separate launches: rng chain, per-env problem indices (weighted while weights are set) and reset keys, step
        self.keys.advance()
        derive_env_keys(self.keys.prob_key, self.keys.reset_key, self.num_envs_global, self.env_offset, self.num_envs,
                        self.bank.num_problems, self.new_problem_idx, self.reset_keys,
                        self._cum_weights if weighted else None)
        self.env.step_into(self.bank, self.state, self.state, actions, dict(out, obs=None) if self.gnn_outputs else out,
                           auto_reset=True, new_problem_idx=self.new_problem_idx, reset_keys=self.reset_keys)
        if self.gnn_outputs:          # the GNN input of the state to continue from, as msat_rollout_step_gnn emits it
            self._gnn_dynamic()
        return out

    def _gnn_dynamic(self) -> None:
        """``msat_gnn_dynamic`` of the current state into ``self.out``'s GNN assignment and clause features."""
        _lib.check(self.env._lib.msat_gnn_dynamic(
            self.bank.plan.handle, _ptr(self.bank.data), self.bank.num_problems, _ptr(self.state), self.num_envs,
            _ptr(self.out["gnn_assignment"]), _ptr(self.out["gnn_clause_features"]), _stream_ptr(self.state.device)),
            "msat_gnn_dynamic")

    def _bind(self, name: str, out: Dict[str, Optional[torch.Tensor]], host: Optional[Dict[str, torch.Tensor]] = None,
              num_steps: int = 1, pipe_slot: Optional[Tuple[int, torch.Tensor]] = None) -> _BoundCall:
        """The argument list of the rollout entry point ``name``, in the header's parameter order, bound to the device
        outputs ``out``; ``host`` is the pinned result buffers of the host-buffer entry points, ``num_steps`` the K of
        ``msat_rollout_steps`` and ``pipe_slot`` the ``(slot, actions_dev)`` of ``msat_rollout_step_host_async``.
        Per-call slots, given to the returned call in this order: the action pointer (``actions``; ``actions_host``
        and ``actions_dev`` for ``msat_rollout_step_host``; ``actions_host`` for ``msat_rollout_step_host_async``);
        then ``rng_in``, ``chain_out`` and ``stream``, which the call fills in itself."""
        s, obs = _ptr(self.state), _ptr(out.get("obs"))
        reward, done = out.get("reward"), out.get("done")
        chain = [_RNG_IN, _CHAIN_OUT, self.num_envs_global, self.env_offset]
        results = [_ptr(reward), 0 if reward is None else int(reward.shape[-1]), _ptr(done),
                   0 if done is None else int(done.shape[-1]), _ptr(out.get("solved")),
                   _ptr(out.get("num_unsatisfied")), _ptr(out.get("episode_step"))]
        if host is not None:
            results += [_ptr(host[k]) for k in ("reward", "done", "solved", "num_unsatisfied", "episode_step")]
        pipe = []
        if name == "msat_rollout_step":
            mid = [s, s, _ACTIONS, *chain, obs, *results]
        elif name == "msat_rollout_step_gnn":
            mid = [s, s, _ACTIONS, *chain, _ptr(out["gnn_assignment"]), _ptr(out["gnn_clause_features"]), *results]
        elif name == "msat_rollout_steps":
            mid = [s, s, _ACTIONS, num_steps, *chain, obs, _ptr(out.get("gnn_assignment")),
                   _ptr(out.get("gnn_clause_features")), 1 if out.get("emit_every_step") else 0, *results,
                   _ptr(out.get("newly_satisfied"))]
        elif name == "msat_rollout_step_host":
            mid = [s, _ACTIONS, _ACTIONS, *chain, obs, *results]
        elif name == "msat_rollout_step_host_async":
            slot_idx, actions_dev = pipe_slot
            pipe = [self._pipe, int(slot_idx)]
            mid = [s, _ACTIONS, _ptr(actions_dev), *chain, obs, *results]
        args = [*pipe, self.bank.plan.handle, _ptr(self.bank.data), self.bank.num_problems, *mid, self.num_envs,
                _STREAM]
        return _BoundCall(getattr(self.env._lib, name), name, args, self.keys, self.state.device)

    def sample_actions(self, logits: torch.Tensor, actions: Optional[torch.Tensor] = None,
                       log_prob: Optional[torch.Tensor] = None):
        """The joint action of the next ``step`` drawn on the device with that step's act_key (learner:397-403):
        ``logits`` float32 ``[B, A, V+1]`` (action mode 0) or ``[B, A, V, 2]`` (mode 1) for this shard's envs ->
        ``(actions, log_prob)`` of shape ``[B, A]`` / ``[B, A, V]``, ready for ``step``.  Rows are indexed in the global
        batch, so every sharding draws the single-device actions, and a run resumed from ``state_dict`` draws what
        the uninterrupted run would have drawn.  Contract: ``sampling.sample_actions``."""
        env, B = self.env, self.num_envs
        A, V = env.num_agents, env.max_vars_per_agent
        shape = (B, A, V + 1) if env.action_mode == 0 else (B, A, V, 2)
        if not isinstance(logits, torch.Tensor) or tuple(logits.shape) != shape:
            got = tuple(logits.shape) if isinstance(logits, torch.Tensor) else type(logits).__name__
            raise ValueError(f"logits must be {shape} for action mode {env.action_mode}, got {got}")
        if logits.device != self.state.device:
            raise ValueError(f"logits must be on {self.state.device}, got {logits.device}")
        rows_per_env = A if env.action_mode == 0 else A * V
        # the rng this env's next step advances: act_key = split(rng)[1] (msat_rng_chain's chain_out[2:4])
        return sample_actions(logits, self.keys.chain[0:2], self.num_envs_global * rows_per_env,
                              self.env_offset * rows_per_env, actions, log_prob)

    # ------------------------------------------------------------------ K fused steps
    def alloc_multi_step_outputs(self, num_steps: int, emit_every_step: bool = False) -> Dict[str, torch.Tensor]:
        """Output buffers of ``steps``: reward / done / info rows ``[K, B, ...]``; the policy input (local
        observations or, with ``gnn_outputs``, the dynamic GNN input) for every step or for the final state."""
        env, dev, B, K = self.env, self.state.device, self.num_envs, int(num_steps)
        d = self.bank.plan.dims
        rc, dc = int(self.out["reward"].shape[-1]), int(self.out["done"].shape[-1])
        lead = (K, B) if emit_every_step else (B,)
        out = {"reward": torch.empty((K, B, rc), dtype=torch.float32, device=dev),
               "done": torch.empty((K, B, dc), dtype=torch.uint8, device=dev),
               "solved": torch.empty((K, B), dtype=torch.uint8, device=dev),
               "num_unsatisfied": torch.empty((K, B), dtype=torch.int32, device=dev),
               "episode_step": torch.empty((K, B), dtype=torch.int32, device=dev),
               "newly_satisfied": (torch.empty((K, B), dtype=torch.int32, device=dev)
                                   if env.reward_mode == "shaped" else None),
               "obs": None, "gnn_assignment": None, "gnn_clause_features": None,
               "emit_every_step": bool(emit_every_step)}
        if self.gnn_outputs:
            out["gnn_assignment"] = torch.empty(lead + (d.n,), dtype=torch.int32, device=dev)
            out["gnn_clause_features"] = torch.empty(lead + (d.m, 3), dtype=torch.float32, device=dev)
        elif self.out.get("obs") is not None:
            out["obs"] = obs_empty(lead + (d.A, d.D), self.env.obs_dtype, dev)
        return out

    def steps(self, actions: torch.Tensor, out: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
        """K rollout steps in ONE launch (``msat_rollout_steps``) for an action table ``[K, B, A(, V)]`` that
        does not depend on the intermediate observations (replay, open-loop evaluation, launch-bound small
        batches).  Identical results to K calls of ``step``; ``out`` from ``alloc_multi_step_outputs``."""
        self._require_plain_resets("steps()")
        self._bind("msat_rollout_steps", out, num_steps=int(actions.shape[0]))(actions.data_ptr())
        return out

    def set_episode_steps(self, steps: torch.Tensor) -> None:
        """Overwrite the per-env ``state.step`` counters (int32 ``[B]``).  Used to de-phase a freshly reset
        batch so that episodes time out at different rollout steps (steady-state auto-reset rate
        ~ B / max_steps per step) instead of all at once."""
        aw = (self.env.num_vars + 31) // 32
        self.state[:, aw].copy_(steps.to(device=self.state.device, dtype=torch.int32))

    # ------------------------------------------------------------------ host-buffer stepping
    def alloc_host_io(self) -> Dict[str, torch.Tensor]:
        """Pinned host buffers for ``step_host``: the action batch in, reward/done/info out (same column
        counts as the device outputs)."""
        env, B = self.env, self.num_envs
        act_shape = (B, env.num_agents) if env.action_mode == 0 else (B, env.num_agents, env.max_vars_per_agent)
        host = env.alloc_step_outputs(B, compact=self.out["reward"].shape[-1] == 1, pinned_host=True)
        host["actions"] = torch.zeros(act_shape, dtype=torch.int32, pin_memory=True)
        return host

    def step_host(self, host: Dict[str, torch.Tensor], actions_dev: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        """End-to-end rollout step for a host-side caller (``msat_rollout_step_host``): host actions are
        copied to the device, the fused step runs, reward/done/info are copied back and the stream is
        synchronised.  Observations stay in HBM (``self.out['obs']``) where the policy consumes them.
        With ``compact_outputs`` the per-agent reward / done values (identical for all agents, env:196,260)
        travel once per env; ``host_views`` expands them without copying."""
        self._require_plain_resets("step_host()")
        if actions_dev is None:
            if not hasattr(self, "_actions_dev"):
                self._actions_dev = torch.empty(host["actions"].shape, dtype=torch.int32, device=self.state.device)
            actions_dev = self._actions_dev
        call, reward, obs = self._host_args or (None, None, None)
        if call is None or reward is not host["reward"] or obs is not self.out["obs"]:
            call = self._bind("msat_rollout_step_host", self.out, host)
            self._host_args = (call, host["reward"], self.out["obs"])
        call(host["actions"].data_ptr(), actions_dev.data_ptr())
        return host

    def alloc_async_io(self, depth: int = 2):
        """Slots of the double-buffered host pipeline: per slot pinned host buffers (actions in, results out),
        a device action staging buffer and device result buffers.  Returns a list of slot dicts."""
        if getattr(self, "_pipe", None) is None:
            h = C.c_void_p()
            _lib.check(self.env._lib.msat_host_pipe_create(C.byref(h), int(depth)), "msat_host_pipe_create")
            self._pipe = h
            self._pipe_depth = int(depth)
        slots = []
        compact = self.out["reward"].shape[-1] == 1
        for _ in range(self._pipe_depth):
            host = self.alloc_host_io()
            dev_out = self.env.alloc_step_outputs(self.num_envs, self.bank.plan.dims, want_obs=False, compact=compact)
            dev_out["obs"] = self.out["obs"]
            slots.append({"host": host, "dev": dev_out,
                          "actions_dev": torch.empty(host["actions"].shape, dtype=torch.int32, device=self.state.device)})
        return slots

    def step_host_async(self, slot_idx: int, slot: Dict, actions_host: Optional[torch.Tensor] = None) -> None:
        """Enqueue one rollout step for host buffers without blocking (``msat_rollout_step_host_async``): the
        action upload, the fused step and the result download of this call overlap the neighbouring steps'.
        ``actions_host`` (pinned; default ``slot['host']['actions']``) must stay untouched until the step's
        kernel has run; read the results from ``slot['host']`` after ``host_wait(slot_idx)``."""
        self._require_plain_resets("step_host_async()")
        call = slot.get("_call")
        if call is None:   # every buffer of a slot is fixed: bound on the slot's first step
            call = slot["_call"] = self._bind("msat_rollout_step_host_async", slot["dev"], slot["host"],
                                              pipe_slot=(slot_idx, slot["actions_dev"]))
        call((slot["host"]["actions"] if actions_host is None else actions_host).data_ptr())

    def host_wait(self, slot_idx: int) -> None:
        """Block until the results of the step last enqueued on this slot are in its host buffers."""
        _lib.check(self.env._lib.msat_host_wait(self._pipe, int(slot_idx)), "msat_host_wait")

    def close(self) -> None:
        if getattr(self, "_pipe", None) is not None:
            self.env._lib.msat_host_pipe_destroy(self._pipe)
            self._pipe = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def host_views(self, host: Dict[str, torch.Tensor]):
        """Reference-shaped dicts over the host buffers: rewards / dones keyed by agent (+ "__all__"),
        as zero-copy views (every agent's value is the same scalar, env:196,260).  The views alias the
        persistent pinned buffers, so they are built once and stay valid across steps."""
        cached = getattr(self, "_host_views", None)
        if cached is not None and cached[0] is host["reward"]:
            return cached[1]
        env = self.env
        rew, done = host["reward"], host["done"].view(torch.bool)
        rewards = {a: rew[:, i if rew.shape[1] > 1 else 0] for i, a in enumerate(env.agents)}
        dones = {a: done[:, i if done.shape[1] > 1 else 0] for i, a in enumerate(env.agents)}
        dones["__all__"] = done[:, -1]
        infos = {"solved": host["solved"].view(torch.bool), "num_unsatisfied": host["num_unsatisfied"],
                 "episode_step": host["episode_step"]}
        self._host_views = (host["reward"], (rewards, dones, infos))
        return self._host_views[1]

    def sat_state(self) -> SATState:
        return SATState(self.env, self.bank, self.state, True)

    # ------------------------------------------------------------------ state import / checkpoints
    def import_state(self, problem_idx, variable_assignments, step=None, done=None,
                     validate: bool = True) -> Optional[torch.Tensor]:
        """Put this shard's envs onto the given states (rows in shard order; leaves as ``SATEnv.import_state``) and
        write the policy input this env emits: ``out["obs"]`` when it is allocated and, with ``gnn_outputs``, the
        GNN assignment / clause features.  The rng chain is not touched."""
        out = self.out
        obs, _ = self.env.import_state(self.bank, problem_idx, variable_assignments, step, done, state_out=self.state,
                                       obs_out=out["obs"], want_obs=out["obs"] is not None, validate=validate)
        if self.gnn_outputs:
            self._gnn_dynamic()
        return obs

    def _signature(self) -> Dict[str, int]:
        env = self.env
        return {"num_vars": env.num_vars, "num_clauses": env.num_clauses, "k": self.bank.k,
                "num_agents": env.num_agents, "num_problems": self.bank.num_problems}

    def state_dict(self) -> Dict:
        """Portable checkpoint of this shard (host tensors, ``torch.save``-able): its rows as reference-shaped
        leaves (``variable_assignments`` [B,n], ``step`` [B], ``done`` [B,A], ``problem_idx`` [B]), the rollout rng
        chain (``RolloutKeys.chain``, 10 words), ``env_offset``, ``num_envs_global`` and a shape ``signature``.
        The packed layout never leaves the process, so the checkpoint loads into either clause-update mode, any
        observation dtype and any later library version.  While problem weights are set, their quantised values are
        stored under ``problem_weights``, and while start states are set, their tables under ``start_states``
        (``words``, ``flip_thr``, ``has_start``); the saved states are those after the starts were applied.
        Synchronises the stream."""
        st = self.sat_state()
        sd = {"variable_assignments": st.variable_assignments.cpu(), "step": st.step.cpu(), "done": st.done.cpu(),
              "problem_idx": st.problem_idx.cpu(), "rng_chain": self.keys.chain.cpu().clone(),
              "env_offset": self.env_offset, "num_envs_global": self.num_envs_global, "signature": self._signature()}
        if self._weights is not None:
            sd["problem_weights"] = self._weights.clone()
        if self._start is not None:
            sd["start_states"] = dict(self._start._asdict())
        return sd

    def load_state_dict(self, sd: Dict) -> Optional[torch.Tensor]:
        """Continue from a checkpoint of ``state_dict``: any dict with this env's signature and global batch size
        whose rows cover this shard's global range ``[env_offset, env_offset + num_envs)``.  Problem indices and
        reset keys depend only on (rng, global env index, global batch size) (DESIGN.md section 7), so a world-1
        checkpoint loads into every rank of a world-N run, and rank checkpoints joined with
        ``merge_state_dicts`` load into any world size, with the values of an uninterrupted single-device run.
        The problem weights and start states are restored too: those of the checkpoint, or the uniform draw / random
        starts for a checkpoint without them.  Returns the policy input written by ``import_state``."""
        sig = {k: int(v) for k, v in dict(sd["signature"]).items()}
        if sig != self._signature():
            raise ValueError(f"checkpoint signature {sig} does not match this env's {self._signature()}")
        if int(sd["num_envs_global"]) != self.num_envs_global:
            raise ValueError(f"checkpoint of {int(sd['num_envs_global'])} envs, this run has {self.num_envs_global}")
        off, rows = int(sd["env_offset"]), int(sd["variable_assignments"].shape[0])
        lo = self.env_offset - off
        if lo < 0 or lo + self.num_envs > rows:
            raise ValueError(f"checkpoint rows [{off}, {off + rows}) do not cover this shard's "
                             f"[{self.env_offset}, {self.env_offset + self.num_envs})")
        weights = sd.get("problem_weights")
        q = None if weights is None else problem_weights(weights, self.bank.num_problems)
        if q is not None and not torch.equal(q, torch.as_tensor(weights, dtype=torch.int64)):
            raise ValueError("checkpoint problem_weights are not quantised weights (problem_weights)")
        starts = _start_table_of(sd)
        if starts is not None and (tuple(starts.words.shape) != (self.bank.num_problems, (self.env.num_vars + 31) // 32)
                                   or tuple(starts.flip_thr.shape) != (self.bank.num_problems,)
                                   or tuple(starts.has_start.shape) != (self.bank.num_problems,)):
            raise ValueError("checkpoint start_states do not match this env's bank")
        rows_of = lambda name: torch.as_tensor(sd[name])[lo:lo + self.num_envs]
        obs = self.import_state(rows_of("problem_idx"), rows_of("variable_assignments"), rows_of("step"),
                                rows_of("done"), validate=True)
        self.keys.chain.copy_(as_u32_tensor(sd["rng_chain"], self.state.device).reshape(10))
        if q is None:
            self._weights = None
        else:
            self._install_weights(q)
        if starts is None:
            self._start = None
        else:
            self._install_starts(starts)
        return obs


def _start_table_of(sd: Dict) -> Optional[StartTable]:
    t = sd.get("start_states")
    if t is None:
        return None
    return StartTable(torch.as_tensor(t["words"], dtype=torch.int32), torch.as_tensor(t["flip_thr"], dtype=torch.int64),
                      torch.as_tensor(t["has_start"], dtype=torch.uint8))


def merge_state_dicts(dicts) -> Dict:
    """Join ``VecSATEnv.state_dict()`` checkpoints of adjacent shards of one run into one (rows in ``env_offset``
    order), e.g. every rank's, which then loads into any world size.  Shards must agree on the problem weights
    (all without, or all with equal ``problem_weights``) and on the start states (all without, or all with equal
    ``start_states`` tables)."""
    dicts = sorted(dicts, key=lambda sd: int(sd["env_offset"]))
    first = dicts[0]
    end = int(first["env_offset"])
    weights = first.get("problem_weights")
    for sd in dicts:
        if int(sd["env_offset"]) != end:
            raise ValueError(f"shards are not adjacent: a gap or overlap at env {end}")
        if dict(sd["signature"]) != dict(first["signature"]) or int(sd["num_envs_global"]) != int(first["num_envs_global"]):
            raise ValueError("checkpoints of different runs")
        if not torch.equal(torch.as_tensor(sd["rng_chain"]), torch.as_tensor(first["rng_chain"])):
            raise ValueError("checkpoints taken at different rollout steps (rng chains differ)")
        w = sd.get("problem_weights")
        if (w is None) != (weights is None) or (w is not None and not torch.equal(torch.as_tensor(w),
                                                                                   torch.as_tensor(weights))):
            raise ValueError("shards have different problem weights")
        st, st0 = _start_table_of(sd), _start_table_of(first)
        if (st is None) != (st0 is None) or (st is not None and not all(torch.equal(x, y) for x, y in zip(st, st0))):
            raise ValueError("shards have different start states")
        end += int(sd["variable_assignments"].shape[0])
    merged = {k: torch.cat([torch.as_tensor(sd[k]) for sd in dicts])
              for k in ("variable_assignments", "step", "done", "problem_idx")}
    merged.update(rng_chain=torch.as_tensor(first["rng_chain"]).clone(), env_offset=int(first["env_offset"]),
                  num_envs_global=int(first["num_envs_global"]), signature=dict(first["signature"]))
    if weights is not None:
        merged["problem_weights"] = torch.as_tensor(weights).clone()
    starts = _start_table_of(first)
    if starts is not None:
        merged["start_states"] = {k: v.clone() for k, v in starts._asdict().items()}
    return merged


class RolloutBuffer:
    """``Transition`` storage (learner:358-369,467-478) for T steps of B envs, laid out ``[T, B, ...]`` so
    the step kernel writes each step's slice in place (no stacking pass).  Observations are *not*
    stored: the packed state (32 B/env at uf100-430) is, and ``SATEnv.get_obs`` regenerates the obs of
    any stored step on demand (the reference stores 63 KB/env-step of obs)."""

    def __init__(self, env: SATEnv, bank: FormulaBank, num_steps: int, num_envs: int):
        dev = env._require_cuda()
        d = bank.plan.dims
        T, B, A = num_steps, num_envs, env.num_agents
        act_shape = (T, B, A) if env.action_mode == 0 else (T, B, A, env.max_vars_per_agent)
        self.env, self.bank, self.num_steps, self.num_envs = env, bank, T, B
        self.state = torch.empty((T, B, d.state_words), dtype=torch.int32, device=dev)     # pre-step state
        self.action = torch.empty(act_shape, dtype=torch.int32, device=dev)
        self.reward = torch.empty((T, B, 1), dtype=torch.float32, device=dev)                # team reward (agent 0)
        self.done = torch.empty((T, B, 1), dtype=torch.uint8, device=dev)                  # global_done only
        self.solved = torch.empty((T, B), dtype=torch.uint8, device=dev)
        self.num_unsatisfied = torch.empty((T, B), dtype=torch.int32, device=dev)
        self.episode_step = torch.empty((T, B), dtype=torch.int32, device=dev)
        self.value = torch.zeros((T, B), dtype=torch.float32, device=dev)
        self.log_prob = torch.zeros(act_shape, dtype=torch.float32, device=dev)

    def step_outputs(self, t: int, obs: Optional[torch.Tensor]) -> Dict[str, Optional[torch.Tensor]]:
        return {"obs": obs, "reward": self.reward[t], "done": self.done[t], "solved": self.solved[t],
                "num_unsatisfied": self.num_unsatisfied[t], "episode_step": self.episode_step[t]}

    @property
    def global_done(self) -> torch.Tensor:
        """``Transition.global_done`` = done["__all__"] (learner:468), dense uint8 ``[T, B]``."""
        return self.done[:, :, 0]

    @property
    def reward_per_agent(self) -> torch.Tensor:
        """``Transition.reward`` ``[T, B, A]`` (learner:471) as a broadcast view of the team reward: every
        agent's reward is the same scalar (env:193-196)."""
        return self.reward.expand(self.num_steps, self.num_envs, self.env.num_agents)

    @property
    def info(self) -> Dict[str, torch.Tensor]:
        """``Transition.info`` (learner:475; env:278-282), ``[T, B]`` each."""
        return {"solved": self.solved.view(torch.bool), "num_unsatisfied": self.num_unsatisfied,
                "episode_step": self.episode_step}

    def problem_stats(self, stats: Optional[torch.Tensor] = None, group=None) -> torch.Tensor:
        """``curriculum.problem_stats`` of this rollout, with each row's problem read from the problem-index word of
        its pre-step state (the episode that ends at step t started on that problem) through strides, without a
        copy.  int64 ``[P, 4]``; added to ``stats`` when given; summed over ranks under ``torch.distributed``."""
        pidx = self.state[:, :, (self.env.num_vars + 31) // 32 + 1]      # state words: assignment, step, problem index
        return problem_stats(pidx, self.global_done, self.solved, self.num_unsatisfied, self.episode_step,
                             self.bank.num_problems, stats, group)

    def pre_step_state(self, t: int) -> SATState:
        """The state the policy acted on at step t (source of ``Transition.local_obs`` / ``global_state`` /
        ``agent_*_masks``, learner:386-387,473-474)."""
        return SATState(self.env, self.bank, self.state[t], True)

    def local_obs(self, t: int) -> torch.Tensor:
        """Observations the policy saw at step t (``Transition.local_obs``, learner:473)."""
        return self.env.get_obs_array(self.pre_step_state(t))

    def collect(self, vec: "VecSATEnv", policy_fn) -> None:
        """``lax.scan(_env_step, carry, None, NUM_STEPS)`` (learner:383-495) for this shard: for each step the
        pre-step state is recorded, ``policy_fn(t, vec) -> (actions, value | None, log_prob | None)`` is
        asked for the joint action (device tensors; it may read ``vec.out['obs']`` / ``vec.state`` and the
        sampling key ``vec.keys`` will hold after this step is ``act_key``), and the fused step writes
        reward / done / info of step t straight into row t of this buffer (pre-reset values, learner:467-478).
        Everything is enqueue-only on the current stream."""
        if vec.num_envs != self.num_envs:
            raise ValueError(f"buffer holds {self.num_envs} envs, the vectorised env {vec.num_envs}")
        obs = vec.out.get("obs")
        for t in range(self.num_steps):
            self.state[t].copy_(vec.state)
            actions, value, log_prob = policy_fn(t, vec)
            self.action[t].copy_(actions.reshape(self.action[t].shape))
            if value is not None:
                self.value[t].copy_(value)
            if log_prob is not None:
                self.log_prob[t].copy_(log_prob.reshape(self.log_prob[t].shape))
            vec.step(self.action[t], out=self.step_outputs(t, obs))
