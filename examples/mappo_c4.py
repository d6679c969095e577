#!/usr/bin/env python
"""BASELINE config 4 end to end: uf250-1065, 16,384 envs sharded over the GPUs of one box, full MAPPO
train cycle -- T-step rollout into the RolloutBuffer (fused step kernel, no step-path collective), GAE with
fused statistics, globally normalised advantages (NCCL all-reduce of 24 bytes), rollout metrics (40 bytes),
PPO epochs on a small MLP actor/critic with DistributedDataParallel (NCCL gradient all-reduce).

    python examples/mappo_c4.py --updates 2                                    # one GPU
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29511 \
        examples/mappo_c4.py --updates 2

Rank 0 prints one JSON line: updates/s, env-steps/s of the whole cycle, the rollout / GAE / update split
(max over ranks, CUDA events) and the bus bandwidth of a gradient-sized NCCL all-reduce.

``--curriculum`` chooses which formulas auto-reset draws:
  none      uniform over the bank (the default, the reference's randint);
  unsolved  per-problem statistics of every rollout are accumulated (``RolloutBuffer.problem_stats``) and after each
            update the weights become ``unsolved_weights`` of the totals;
  walksat   one WalkSAT call over a reset of every bank formula labels the formulas it solves; only those are drawn.
  reverse   the walksat draw, and every episode starts at its formula's WalkSAT solution with each bit flipped with
            probability q (``set_start_states``; q starts at --start-flip-prob).  After every update
            ``adapt_flip_prob`` moves each formula's q with that rollout's solve rate: up where the policy solves
            it, down where it does not (a reverse curriculum).
The JSON line then also reports the share of the bank solved at least once during the timed updates (and, for
reverse, the mean q and the share of formulas at q_max).
Reference structure: src/learners/mappo_gnn_sat_learner.py:381-732, configs/MAPPO_CONFIG.yaml:27-48.
"""
import argparse
import json
import os
import sys
import time
from pathlib import Path

import torch
import torch.distributed as dist

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import marl_sat_b200 as M                                           # noqa: E402
from marl_sat_b200 import synth                                     # noqa: E402
from marl_sat_b200.curriculum import adapt_flip_prob                 # noqa: E402
from marl_sat_b200.mappo import MAPPOTrainer, MLPActorCritic, PPOConfig    # noqa: E402

Q_MAX = 0.5          # adapt_flip_prob's default ceiling: a start as random as the reference's draw


def walksat_solvable(M, env, bank, max_flips, dev):
    """bool [P]: the formulas one WalkSAT call (noise 0.5) solves from a reset of every bank formula, and int32 [P, n]
    the searched assignments (row p is formula p; a solution where solved)."""
    P = bank.num_problems
    idx = torch.arange(P, dtype=torch.int32, device=dev)
    keys = M.env.as_u32_tensor(torch.stack([torch.zeros(P, dtype=torch.int64), torch.arange(P)], 1), dev)
    _, state = env.reset_from_bank(bank, idx, keys, want_obs=False)
    res = M.walksat(state, keys, max_flips)
    solved = res.solved.cpu()
    if not bool(solved.any()):
        raise SystemExit(f"WalkSAT solved none of the {P} formulas in {max_flips} flips: nothing to train on")
    return solved, res.state.variable_assignments


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=250)
    ap.add_argument("--m", type=int, default=1065)
    ap.add_argument("--envs", type=int, default=16384, help="global env count (sharded over the ranks)")
    ap.add_argument("--problems", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=512, help="NUM_STEPS of the rollout (MAPPO_CONFIG.yaml:30)")
    ap.add_argument("--max-steps", type=int, default=512)
    ap.add_argument("--epochs", type=int, default=4)
    ap.add_argument("--minibatch", type=int, default=16384, help="env-steps per minibatch per rank")
    ap.add_argument("--updates", type=int, default=2)
    ap.add_argument("--hidden", type=int, default=128)
    ap.add_argument("--obs-int8", action="store_true",
                    help="int8 observations (MSAT_OBS_INT8): same values, a quarter of the bytes the policy reads")
    ap.add_argument("--curriculum", choices=("none", "unsolved", "walksat", "reverse"), default="none",
                    help="problem draw of auto-reset: uniform, weighted by unsolved rate, or WalkSAT-solved formulas "
                         "only; reverse also starts episodes near the WalkSAT solutions")
    ap.add_argument("--start-flip-prob", type=float, default=0.05,
                    help="initial per-bit flip probability q of the reverse curriculum's starts")
    ap.add_argument("--walksat-flips", type=int, default=10000, help="flip budget of the walksat curriculum's labelling")
    ap.add_argument("--act-key-sampling", action="store_true",
                    help="draw actions on the device with each step's act_key (msat_sample_actions): trajectories "
                         "independent of the world size")
    args = ap.parse_args()

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    env = M.SATEnv(args.n, args.m, args.max_steps, verbose=False, device=dev,
                   obs_dtype=torch.int8 if args.obs_int8 else torch.int32)
    problems = synth.uniform_ksat_torch(args.problems, args.n, args.m, 3, seed=20261018 + 4, device=dev)
    bank = env.make_bank(problems, validate=False)
    vec = M.VecSATEnv(env, bank, args.envs, M.prng_key(42), world_size=world, rank=rank, compact_outputs=True)
    labelled = solutions = flip_prob = None
    if args.curriculum in ("walksat", "reverse"):
        labelled, solutions = walksat_solvable(M, env, bank, args.walksat_flips, dev)
        vec.set_problem_weights(labelled)           # identical on every rank: same bank, same keys
    if args.curriculum == "reverse":
        flip_prob = torch.full((bank.num_problems,), float(args.start_flip_prob), dtype=torch.float64)
        vec.set_start_states(solutions, flip_prob, has_start=labelled)
    vec.reset()
    torch.manual_seed(0)                       # identical initial weights on every rank
    net = MLPActorCritic(env, hidden=args.hidden)
    cfg = PPOConfig(num_steps=args.steps, update_epochs=args.epochs, minibatch_size=args.minibatch)
    trainer = MAPPOTrainer(vec, net, cfg, seed=1, act_key_sampling=args.act_key_sampling)

    trainer.train_cycle()                      # warm-up cycle (allocator, cuBLAS handles, NCCL channels)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    last = None
    split = torch.zeros(3, dtype=torch.float64, device=dev)
    totals = torch.zeros((bank.num_problems, 4), dtype=torch.int64, device=dev)     # all-reduced per-problem stats
    for _ in range(args.updates):
        last = trainer.train_cycle()
        if args.curriculum != "none":
            trainer.buf.problem_stats(totals)   # this rollout's counters, summed over the ranks, added to the totals
        if args.curriculum == "unsolved":
            vec.set_problem_weights(M.unsolved_weights(totals))
        if args.curriculum == "reverse":              # this rollout's rates, identical on every rank
            flip_prob = adapt_flip_prob(trainer.buf.problem_stats(), flip_prob)
            vec.set_start_states(solutions, flip_prob, has_start=labelled)
        split += torch.tensor([last["rollout_ms"], last["gae_metrics_ms"], last["update_ms"]], dtype=torch.float64,
                              device=dev)
    torch.cuda.synchronize()
    wall = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(wall, op=dist.ReduceOp.MAX)
        dist.all_reduce(split, op=dist.ReduceOp.MAX)
    bus = trainer.gradient_allreduce_busbw()
    # replicas must still be identical after the updates
    flat = torch.cat([p.detach().reshape(-1) for p in trainer.raw_net.parameters()])
    ref = flat.clone()
    if world > 1:
        dist.broadcast(ref, src=0)
    in_sync = bool(torch.equal(flat, ref))
    if world > 1:
        ok = torch.tensor([1 if in_sync else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        in_sync = bool(ok.item())
    if rank == 0:
        t = float(wall.item())
        rollout_ms, gae_ms, update_ms = (split / args.updates).tolist()
        print(json.dumps({
            "what": "BASELINE config 4: full MAPPO train cycle (rollout + GAE + PPO update)",
            "config": {"n": args.n, "m": args.m, "envs_global": args.envs, "envs_per_gpu": vec.num_envs,
                       "num_steps": args.steps, "update_epochs": args.epochs, "minibatch_per_rank": args.minibatch,
                       "agents": env.num_agents, "obs_dim": env.obs_dim, "policy": f"MLP actor/critic, hidden {args.hidden}",
                       "params": sum(p.numel() for p in net.parameters())},
            "n_gpus": world, "updates": args.updates, "updates_per_s": args.updates / t,
            "env_steps_per_s": args.updates * args.steps * args.envs / t,
            "ms_per_update": {"rollout": rollout_ms, "gae_normalise_metrics": gae_ms, "ppo_update": update_ms,
                              "wall": 1e3 * t / args.updates},
            "rollout_env_steps_per_s": args.steps * args.envs / (rollout_ms * 1e-3),
            "gradient_allreduce": bus, "replicas_in_sync": in_sync,
            "metrics_last_update": {k: v for k, v in last.items() if not k.endswith("_ms")},
            "curriculum": args.curriculum,
            "bank_share_solved_at_least_once": (None if args.curriculum == "none"
                                                else float((totals[:, 1] > 0).double().mean())),
            "bank_share_walksat_solved": None if labelled is None else float(labelled.double().mean()),
            "start_flip_prob_mean": (None if flip_prob is None
                                     else float(flip_prob[labelled].mean())),
            "start_share_at_q_max": (None if flip_prob is None
                                     else float((flip_prob[labelled] >= Q_MAX).double().mean())),
        }))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if not in_sync:
        raise SystemExit("replicas diverged")


if __name__ == "__main__":
    main()
