"""MAPPO train cycle around the B200-native env path: rollout -> GAE -> PPO update, data-parallel over GPUs.

Mirrors the structure of ``make_train_cycle`` in the reference learner
(``/root/reference/src/learners/mappo_gnn_sat_learner.py:381-732``, cited as learner:LINE):

    rollout        ``lax.scan(_env_step, ..., NUM_STEPS)``                 learner:383-495   -> ``RolloutBuffer.collect``
    last value     critic on the final state                                learner:497-502
    GAE            ``_calculate_gae`` + global normalisation                learner:504-532   -> ``calculate_gae`` / ``normalize_advantages``
    PPO epochs     shuffle, minibatches, clipped actor / value loss         learner:563-660   -> ``ppo_loss`` + torch autograd
    metrics        episodic return, solve rate, ...                         learner:661-686   -> ``rollout_metrics``

The environments (and with them the rollout buffer) are sharded across ranks with no collective on the step
path; the only collectives are the 24-byte all-reduce of the advantage statistics, the 40-byte all-reduce of
the metric sums and the NCCL gradient all-reduce of the update (``DistributedDataParallel``) -- the reference
itself is single-device, so the sharded update differs from it only by reduction order.

The networks are ordinary PyTorch modules and deliberately small (north_star: "the small actor/critic MLPs
remain ordinary" framework code): a shared per-agent MLP actor on the int32 local observations and an MLP
critic on the global (assignment, clause status) vector.  Observations are never stored: the update
regenerates the observations of each minibatch from the packed pre-step states (32 B instead of 94 KB per
env-step at uf250-1065) with ``msat_get_obs``.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, Optional

import torch
import torch.nn as nn

from .env import SATEnv, SATState
from .features import dynamic_features
from .gae import calculate_gae, normalize_advantages
from .metrics import rollout_metrics
from .rollout import RolloutBuffer, VecSATEnv


@dataclass
class PPOConfig:
    """The ``training`` block of configs/MAPPO_CONFIG.yaml (reference values as defaults)."""
    num_steps: int = 512
    update_epochs: int = 4
    minibatch_size: int = 256           # env-steps per minibatch *per rank*
    learning_rate: float = 1e-4
    gamma: float = 0.995
    gae_lambda: float = 0.95
    clip_eps: float = 0.12
    ent_coef: float = 0.005
    vf_coef: float = 0.5
    vf_clip: float = 0.5


class MLPActorCritic(nn.Module):
    """Shared per-agent actor on the local observation (values in {-1, 0, 1}) plus a learned agent embedding;
    centralised critic on ``[assignment | clause satisfied]``."""

    def __init__(self, env: SATEnv, hidden: int = 128):
        super().__init__()
        A, V, D = env.num_agents, env.max_vars_per_agent, env.obs_dim
        if env.action_mode != 0:
            raise NotImplementedError("the example policy covers action_mode 0 (Discrete(V+1) per agent)")
        self.num_agents, self.num_actions = A, V + 1
        self.agent_embedding = nn.Embedding(A, hidden)
        self.actor_in = nn.Linear(D, hidden)
        self.actor_body = nn.Sequential(nn.ReLU(), nn.Linear(hidden, hidden // 2), nn.ReLU(),
                                        nn.Linear(hidden // 2, V + 1))
        self.critic = nn.Sequential(nn.Linear(env.num_vars + env.num_clauses, hidden), nn.ReLU(),
                                    nn.Linear(hidden, hidden // 2), nn.ReLU(), nn.Linear(hidden // 2, 1))

    def actor_logits(self, obs: torch.Tensor) -> torch.Tensor:
        """obs int32 ``[N, A, D]`` -> logits float32 ``[N, A, V+1]``."""
        x = self.actor_in(obs.to(self.actor_in.weight.dtype))
        x = x + self.agent_embedding.weight[None, :, :]
        return self.actor_body(x).float()

    def value(self, assignment: torch.Tensor, clause_sat: torch.Tensor) -> torch.Tensor:
        """assignment int32 ``[N, n]``, clause_sat float ``[N, m]`` -> value float32 ``[N]``."""
        g = torch.cat([assignment.to(clause_sat.dtype), clause_sat], dim=-1)
        return self.critic(g).squeeze(-1).float()

    def forward(self, obs, assignment, clause_sat):
        return self.actor_logits(obs), self.value(assignment, clause_sat)


def ppo_loss(logits: torch.Tensor, value: torch.Tensor, action: torch.Tensor, old_log_prob: torch.Tensor,
             old_value: torch.Tensor, advantages: torch.Tensor, targets: torch.Tensor, cfg: PPOConfig,
             ent_coef: Optional[float] = None):
    """``_loss_fn`` of learner:595-646 for action_mode 0: per-agent ratios against the shared (already
    normalised) team advantage, clipped value loss, entropy bonus.  Returns ``(total, (value_loss, actor_loss,
    entropy))``."""
    dist = torch.distributions.Categorical(logits=logits)
    log_prob = dist.log_prob(action.long())                                   # learner:610
    ratio = torch.exp(log_prob - old_log_prob)                                # learner:611-612
    gae = advantages[:, None]                                                 # learner:614
    loss_actor1 = ratio * gae                                                 # learner:619
    loss_actor2 = torch.clamp(ratio, 1.0 - cfg.clip_eps, 1.0 + cfg.clip_eps) * gae
    loss_actor = -torch.minimum(loss_actor1, loss_actor2).mean()              # learner:636
    entropy = dist.entropy().mean()                                           # learner:637
    coef = cfg.ent_coef if ent_coef is None else ent_coef
    actor_loss = loss_actor - coef * entropy                                  # learner:638
    value_pred_clipped = old_value + (value - old_value).clamp(-cfg.vf_clip, cfg.vf_clip)   # learner:639-640
    value_losses = (value - targets) ** 2
    value_losses_clipped = (value_pred_clipped - targets) ** 2
    value_loss = 0.5 * torch.maximum(value_losses, value_losses_clipped).mean()             # learner:641-643
    total = actor_loss + cfg.vf_coef * value_loss                             # learner:644
    return total, (value_loss, loss_actor, entropy)


class MAPPOTrainer:
    """One process per GPU.  ``vec`` is this rank's shard of the env batch; ``net`` is wrapped in
    ``DistributedDataParallel`` when ``torch.distributed`` is initialised with more than one rank.

    ``act_key_sampling=True`` draws the rollout's actions on the device with each step's act_key
    (``VecSATEnv.sample_actions``, learner:397-403): the trajectories then depend only on the seed key, the network
    and the global batch, not on the world size, and a run resumed from ``VecSATEnv.state_dict`` continues exactly.
    The default draws with ``torch.multinomial`` and a per-rank generator."""

    def __init__(self, vec: VecSATEnv, net: MLPActorCritic, cfg: PPOConfig, seed: int = 0, autocast: bool = True,
                 act_key_sampling: bool = False):
        self.vec, self.cfg = vec, cfg
        self.env = vec.env
        self.device = vec.state.device
        self.raw_net = net.to(self.device)
        self.world = (torch.distributed.get_world_size() if torch.distributed.is_available()
                      and torch.distributed.is_initialized() else 1)
        self.net = self.raw_net
        if self.world > 1:
            self.net = nn.parallel.DistributedDataParallel(self.raw_net, device_ids=[self.device.index])
        self.opt = torch.optim.Adam(self.raw_net.parameters(), lr=cfg.learning_rate, eps=1e-5)
        self.buf = RolloutBuffer(self.env, vec.bank, cfg.num_steps, vec.num_envs)
        self.gen = torch.Generator(device=self.device).manual_seed(seed + 7919 * vec.env_offset)
        self.autocast = autocast
        self.act_key_sampling = act_key_sampling

    # -- the critic's global input from a packed state -------------------------------------------------------
    def _global_features(self, state: SATState):
        assignment, cf = dynamic_features(state)
        return assignment, cf[:, :, 0]

    @torch.no_grad()
    def _policy(self, t: int, vec: VecSATEnv):
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=self.autocast):
            logits = self.raw_net.actor_logits(vec.out["obs"])
            assignment, sat = self._global_features(vec.sat_state())
            value = self.raw_net.value(assignment, sat)
        if self.act_key_sampling:
            action, log_prob = vec.sample_actions(logits)
            return action, value, log_prob
        probs = torch.softmax(logits, dim=-1)
        action = torch.multinomial(probs.reshape(-1, probs.shape[-1]), 1, generator=self.gen).reshape(probs.shape[:-1])
        log_prob = torch.log(torch.gather(probs, -1, action[..., None]).squeeze(-1).clamp_min(1e-30))
        return action.to(torch.int32), value, log_prob

    def train_cycle(self) -> Dict[str, float]:
        cfg, vec, buf, dev = self.cfg, self.vec, self.buf, self.device
        T, B = cfg.num_steps, vec.num_envs
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        # ---- 1. rollout (learner:383-495) ----
        buf.collect(vec, self._policy)
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16, enabled=self.autocast):
            last_val = self.raw_net.value(*self._global_features(vec.sat_state()))          # learner:497-502
        ev[1].record()
        # ---- 2. GAE + global normalisation (learner:504-532) ----
        stats = torch.zeros(3, dtype=torch.float64, device=dev)
        advantages, targets = calculate_gae(buf.reward[:, :, 0], buf.global_done, buf.value, last_val, cfg.gamma,
                                            cfg.gae_lambda, stats=stats)
        normalize_advantages(advantages, stats=stats)            # all-reduces (count, sum, sum of squares)
        metrics = rollout_metrics(buf.reward, buf.global_done, buf.solved, buf.num_unsatisfied, buf.episode_step,
                                  num_envs_global=vec.num_envs_global)
        ev[2].record()
        # ---- 3. PPO epochs (learner:563-660) ----
        flat_state = buf.state.reshape(T * B, -1)
        flat_action = buf.action.reshape(T * B, -1)
        flat_logp = buf.log_prob.reshape(T * B, -1)
        flat_value, flat_adv, flat_tgt = buf.value.reshape(-1), advantages.reshape(-1), targets.reshape(-1)
        mb = min(cfg.minibatch_size, T * B)
        num_minibatches = (T * B) // mb
        losses = torch.zeros(3, device=dev)
        steps = 0
        for _ in range(cfg.update_epochs):
            perm = torch.randperm(T * B, device=dev, generator=self.gen)                    # learner:568
            for i in range(num_minibatches):
                idx = perm[i * mb:(i + 1) * mb]
                state = SATState(self.env, vec.bank, flat_state[idx].contiguous(), True)
                obs = self.env.get_obs_array(state)              # Transition.local_obs of these samples (learner:473)
                assignment, sat = self._global_features(state)
                with torch.autocast("cuda", dtype=torch.bfloat16, enabled=self.autocast):
                    logits, value = self.net(obs, assignment, sat)
                total, aux = ppo_loss(logits, value, flat_action[idx], flat_logp[idx], flat_value[idx],
                                      flat_adv[idx], flat_tgt[idx], cfg)
                self.opt.zero_grad(set_to_none=True)
                total.backward()                                 # DDP: NCCL gradient all-reduce overlaps the backward
                self.opt.step()
                losses += torch.stack([a.detach() for a in aux])
                steps += 1
        ev[3].record()
        torch.cuda.synchronize()
        vl, al, ent = (losses / max(steps, 1)).tolist()
        metrics.update({"value_loss": vl, "actor_loss": al, "entropy": ent, "optimizer_steps": steps,
                        "rollout_ms": ev[0].elapsed_time(ev[1]), "gae_metrics_ms": ev[1].elapsed_time(ev[2]),
                        "update_ms": ev[2].elapsed_time(ev[3])})
        return metrics

    def gradient_allreduce_busbw(self, reps: int = 20) -> Optional[Dict[str, float]]:
        """NCCL all-reduce of one gradient-sized buffer, timed with CUDA events: algorithm and bus bandwidth."""
        if self.world <= 1:
            return None
        nbytes = sum(p.numel() * p.element_size() for p in self.raw_net.parameters())
        flat = torch.zeros(nbytes // 4, dtype=torch.float32, device=self.device)
        for _ in range(3):
            torch.distributed.all_reduce(flat)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            torch.distributed.all_reduce(flat)
        e1.record()
        torch.cuda.synchronize()
        t = e0.elapsed_time(e1) * 1e-3 / reps
        return {"bytes": nbytes, "us": t * 1e6, "algbw_gbs": nbytes / t / 1e9,
                "busbw_gbs": nbytes / t / 1e9 * 2 * (self.world - 1) / self.world}
