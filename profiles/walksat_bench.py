"""Throughput of the batched WalkSAT kernel (msat_walksat) from reset states.

Shapes: uf100-430 x 65,536 envs and uf250-1065 x 16,384 envs, one uniform random formula per env, states from
msat_reset, noise 0.5, max_flips 10,000.  Each timed launch searches the same reset states again (the state is
copied back between launches, outside the events); after a warm-up launch the reported time is the median over
`--reps` launches, each between CUDA events on one stream.

Reported per shape: ms per launch, flip iterations executed (the sum of the `flips` output), flips/s, the solved
fraction, and the solved fraction at the env's own budget max_steps x A (max_steps 512, the reference
configuration): envs solved within that many flips, read from the `flips` output.  The kernel works out of shared
memory and is bound by instruction issue, not by HBM, so no share of a bandwidth peak is stated.

    python profiles/walksat_bench.py [--reps 5] [--out result.json]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

sys.dont_write_bytecode = True
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

MAX_STEPS = 512
SHAPES = [("uf100-430", 100, 430, 65536), ("uf250-1065", 250, 1065, 16384)]


def power_limit() -> str:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return out.stdout.strip() or "unknown"
    except Exception:
        return "unknown"


def run_shape(M, name, n, m, B, max_flips, noise, reps, seed=0):
    from marl_sat_b200.env import _ptr
    from marl_sat_b200.synth import uniform_ksat_torch
    dev = torch.device("cuda")
    env = M.SATEnv(n, m, MAX_STEPS, verbose=False)
    bank = env.make_bank(uniform_ksat_torch(B, n, m, 3, seed=seed, device=dev))
    g = torch.Generator(device=dev).manual_seed(seed)
    idx = torch.arange(B, dtype=torch.int32, device=dev)
    reset_keys = torch.randint(-2 ** 31, 2 ** 31 - 1, (B, 2), generator=g, device=dev, dtype=torch.int64).to(torch.int32)
    keys = torch.randint(-2 ** 31, 2 ** 31 - 1, (B, 2), generator=g, device=dev, dtype=torch.int64).to(torch.int32)
    _, start = env.reset_from_bank(bank, idx, reset_keys, want_obs=False)
    work = start.packed.clone()
    solved = torch.empty(B, dtype=torch.uint8, device=dev)
    flips = torch.empty(B, dtype=torch.int32, device=dev)
    lib, stream = env._lib, torch.cuda.current_stream(dev).cuda_stream

    def launch():
        rc = lib.msat_walksat(bank.plan.handle, _ptr(bank.data), B, _ptr(work), _ptr(keys), max_flips, 0, noise,
                              _ptr(solved), _ptr(flips), B, stream)
        assert rc == 0, rc

    work.copy_(start.packed)
    launch()                                      # warm-up (module load, shared-memory opt-in)
    times = []
    for _ in range(reps):
        work.copy_(start.packed)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        launch()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    # every launch searched the same states with the same keys: the outputs of the last one are the result
    total_flips = int(flips.long().sum())
    budget = MAX_STEPS * env.num_agents
    ok = solved.bool()
    ms = statistics.median(times)
    return {"envs": B, "n": n, "m": m, "num_agents": env.num_agents, "max_flips": max_flips, "noise": noise,
            "ms_per_launch_median": round(ms, 3), "ms_min": round(min(times), 3), "ms_max": round(max(times), 3),
            "flips_executed": total_flips, "flips_per_s": round(total_flips / (ms * 1e-3), 1),
            "solved_fraction": round(float(ok.float().mean()), 5),
            "env_budget_flips": budget,
            "solved_fraction_at_env_budget": round(float((ok & (flips <= budget)).float().mean()), 5)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--max-flips", type=int, default=10000)
    ap.add_argument("--noise", type=float, default=0.5)
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: this measurement has no CPU fallback")
    import marl_sat_b200 as M
    result = {"what": "msat_walksat (WalkSAT/SKC) from msat_reset states", "device": torch.cuda.get_device_name(),
              "power_limit": power_limit(),
              "timing": f"CUDA events around one launch, median over {args.reps} launches after one warm-up launch",
              "shapes": {}}
    for name, n, m, B in SHAPES:
        result["shapes"][name] = run_shape(M, name, n, m, B, args.max_flips, args.noise, args.reps)
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
            f.write("\n")


if __name__ == "__main__":
    main()
