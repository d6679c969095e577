"""Time of the on-device action draw (msat_sample_actions) against the MAPPO trainer's torch sampler on the same logits.

The torch sampler is MAPPOTrainer's default draw: softmax, torch.multinomial with a torch.Generator, gather and log
over the [B, A, V+1] logits.  Shapes (action mode 0, float32 logits of standard-normal values):
  uf100-430 x 65,536 envs   25 agents x 5 classes   (the headline batch)
  uf250-1065 x 16,384 envs  15 agents x 18 classes  (BASELINE config 4)
  uf100-430 x 8,192 envs    one rank's shard of the headline batch on eight GPUs
Each of `--rounds` rounds times `--iters` back-to-back calls of each sampler between CUDA events, the two samplers
alternating inside the round; the reported time per call is the median over the rounds.  The logits (33 MB at the
headline) fit in the 126 MB L2, as they do in a rollout, where the policy has just written them.  Bytes are the
kernel's compulsory traffic (logits read, actions and log-probabilities written); the Threefry blocks are one per
logit element.

    python profiles/sample_actions_bench.py [--rounds 9] [--iters 20] [--out result.json]
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

SHAPES = [("uf100-430 x 65536", 65536, 25, 5), ("uf250-1065 x 16384", 16384, 15, 18),
          ("uf100-430 x 8192 (shard of 65536 on 8 GPUs)", 8192, 25, 5)]
HBM_BYTES_PER_S = 7.7e12          # HGX B200 data sheet, one GPU


def gpu_info() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        name, power, clock = (s.strip() for s in out.stdout.strip().split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception:
        return {"name": torch.cuda.get_device_name(), "power_limit": "unknown", "max_sm_clock": "unknown"}


def torch_sampler(logits: torch.Tensor, gen: torch.Generator):
    """MAPPOTrainer._policy's default draw."""
    probs = torch.softmax(logits, dim=-1)
    action = torch.multinomial(probs.reshape(-1, probs.shape[-1]), 1, generator=gen).reshape(probs.shape[:-1])
    log_prob = torch.log(torch.gather(probs, -1, action[..., None]).squeeze(-1).clamp_min(1e-30))
    return action.to(torch.int32), log_prob


def run_shape(M, B, A, C, rounds, iters):
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(B + C)
    logits = torch.randn((B, A, C), generator=g, device=dev)
    rng = torch.tensor([0, 42], dtype=torch.int32, device=dev)
    actions = torch.empty((B, A), dtype=torch.int32, device=dev)
    log_prob = torch.empty((B, A), dtype=torch.float32, device=dev)
    gen = torch.Generator(device=dev).manual_seed(7)

    def kernel():
        M.sample_actions(logits, rng, actions=actions, log_prob=log_prob)

    def reference():
        torch_sampler(logits, gen)

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / iters

    for fn in (kernel, reference):                # warm-up: module load, allocator, multinomial's workspace
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    t_kernel, t_torch = [], []
    for r in range(rounds):
        order = (kernel, reference) if r % 2 == 0 else (reference, kernel)
        for fn in order:
            (t_kernel if fn is kernel else t_torch).append(timed(fn))
    ms_k, ms_t = statistics.median(t_kernel), statistics.median(t_torch)
    N = B * A * C
    bytes_k = 4 * N + 8 * B * A
    return {"envs": B, "agents": A, "classes": C, "elements": N,
            "msat_sample_actions_us": round(ms_k * 1e3, 2), "torch_sampler_us": round(ms_t * 1e3, 2),
            "speedup": round(ms_t / ms_k, 2),
            "msat_us_min_max": [round(min(t_kernel) * 1e3, 2), round(max(t_kernel) * 1e3, 2)],
            "torch_us_min_max": [round(min(t_torch) * 1e3, 2), round(max(t_torch) * 1e3, 2)],
            "kernel_bytes": bytes_k, "kernel_bytes_per_s": round(bytes_k / (ms_k * 1e-3) / 1e9, 1),
            "kernel_bytes_share_of_hbm_peak": round(bytes_k / (ms_k * 1e-3) / HBM_BYTES_PER_S, 3),
            "threefry_blocks_per_s": round(N / (ms_k * 1e-3) / 1e9, 2)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--rounds", type=int, default=9)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: this measurement has no CPU fallback")
    import marl_sat_b200 as M
    result = {"what": "msat_sample_actions vs MAPPOTrainer's torch sampler (softmax + multinomial + gather + log)",
              "gpu": gpu_info(),
              "timing": f"CUDA events around {args.iters} back-to-back calls; median over {args.rounds} rounds, the "
                        f"two samplers alternating inside each round",
              "bytes_per_s_unit": "GB/s (1e9); the share of peak is against 7.7 TB/s and the logits are L2-resident",
              "shapes": {}}
    for name, B, A, C in SHAPES:
        result["shapes"][name] = run_shape(M, B, A, C, args.rounds, args.iters)
        torch.cuda.empty_cache()
    print(json.dumps(result))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
            f.write("\n")


if __name__ == "__main__":
    main()
