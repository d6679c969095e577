"""Cost of the start states (``msat_apply_start_states``, ``VecSATEnv.set_start_states``).

1. Step cost.  One ``VecSATEnv`` (512-step episodes, de-phased as ``bench.py`` does, so about B / 512 envs restart per
   step) alternates two arms from the same saved state: the fused step alone (random starts) and the fused step
   followed by ``msat_apply_start_states`` (every problem has a start, q = 0.05), each eager (one Python call per step)
   and as a replayed CUDA graph of 32 steps.  Shapes: uf100-430 x 65,536 (headline), its first 8,192-env shard, and
   uf250-1065 x 16,384.  Median / min / max ms per step over the rounds (CUDA events); the arm order alternates.
2. The call alone, on the headline shape and the shard: at the natural reset rate (the de-phased state, ~B / 512 envs
   with step 0) and with every env restarting (all steps 0, as ``max_steps = 1`` leaves them).  The call is
   idempotent on a given state, so repeated launches measure the same work; median over 5 x 200 launches.

    python profiles/start_states_bench.py [--rounds 9] [--steps 192] [--out result.json]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

MAX_STEPS, SEED, ACTION_CYCLE, G, Q = 512, 42, 64, 32, 0.05


def card() -> dict:
    info = {"name": torch.cuda.get_device_name(), "power_limit": "unknown", "max_sm_clock": "unknown"}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in out.stdout.strip().split(",")]
    except Exception:
        pass
    return info


def summary(ms):
    return {"median": statistics.median(ms), "min": min(ms), "max": max(ms), "rounds": ms}


def events_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def setup(M, n, m, Bg, shard):
    from marl_sat_b200 import synth
    dev = torch.device("cuda", torch.cuda.current_device())
    env = M.SATEnv(n, m, MAX_STEPS, verbose=False, device=dev)
    bank = env.make_bank(synth.uniform_ksat_torch(Bg, n, m, 3, seed=20261018 + 2, device=dev), validate=False)
    vec = M.VecSATEnv(env, bank, Bg, M.prng_key(SEED), world_size=shard[0], rank=shard[1])
    starts = torch.randint(0, 2, (bank.num_problems, n), generator=torch.Generator().manual_seed(5), dtype=torch.int32)
    vec.reset()
    g = torch.arange(vec.env_offset, vec.env_offset + vec.num_envs, device=dev, dtype=torch.int64)
    vec.set_episode_steps((g % MAX_STEPS).to(torch.int32))          # bench.py's de-phasing
    return env, bank, vec, starts


def step_cost(M, label, n, m, Bg, shard, rounds, steps):
    env, bank, vec, starts = setup(M, n, m, Bg, shard)
    dev = vec.state.device
    B, A, V = vec.num_envs, env.num_agents, env.max_vars_per_agent
    gen = torch.Generator(device=dev).manual_seed(1234 + shard[1])
    actions = torch.randint(0, V + 1, (ACTION_CYCLE, B, A), generator=gen, device=dev, dtype=torch.int32)
    state0, chain0, cur0 = vec.state.clone(), vec.keys._bufs.clone(), vec.keys._cur

    def restore():
        vec.state.copy_(state0)
        vec.keys._bufs.copy_(chain0)
        vec.keys._cur = cur0

    def arm_starts(arm):
        vec.set_start_states(starts if arm == "starts" else None, Q)

    graphs = {}
    for arm in ("random", "starts"):
        arm_starts(arm)
        restore()
        for i in range(4):
            vec.step(actions[i])
        torch.cuda.synchronize()
        restore()
        graphs[arm] = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graphs[arm]):
            for i in range(G):
                vec.step(actions[i])
        torch.cuda.synchronize()
    launches = steps // G
    res = {"case": label, "envs_global": Bg, "envs_this_gpu": B, "shard": list(shard), "flip_prob": Q}
    for mode in ("eager", "graph"):
        def run(arm):
            arm_starts(arm)
            restore()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            if mode == "eager":
                for i in range(launches * G):
                    vec.step(actions[i % ACTION_CYCLE])
            else:
                for _ in range(launches):
                    graphs[arm].replay()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / (launches * G)

        for arm in ("random", "starts"):
            run(arm)
        ms = {"random": [], "starts": []}
        for r in range(rounds):
            for arm in (("random", "starts") if r % 2 == 0 else ("starts", "random")):
                ms[arm].append(run(arm))
        u, w = summary(ms["random"]), summary(ms["starts"])
        res[mode] = {"ms_per_step": {"random": u, "starts": w},
                     "overhead_ms": w["median"] - u["median"], "overhead_frac": w["median"] / u["median"] - 1.0,
                     "random_spread_ms": u["max"] - u["min"], "starts_spread_ms": w["max"] - w["min"]}
    vec.set_start_states(None)
    del graphs, vec, bank, env
    torch.cuda.empty_cache()
    return res


def call_alone(M, label, n, m, Bg, shard, reps=200):
    env, bank, vec, starts = setup(M, n, m, Bg, shard)
    vec.set_start_states(starts, Q)
    vec.step(torch.zeros((vec.num_envs, env.num_agents), dtype=torch.int32, device=vec.state.device))
    natural = vec.state.clone()
    res = {"case": label, "envs_this_gpu": vec.num_envs}
    aw = (n + 31) // 32
    for name, restarting in (("natural_reset_rate", None), ("every_env_restarts", 0)):
        vec.state.copy_(natural)
        if restarting is not None:
            vec.state[:, aw] = restarting
        fresh = int((vec.state[:, aw] == 0).sum())
        fn = lambda: vec._apply_starts(vec.keys.reset_key, vec.out["obs"])
        for _ in range(10):
            fn()
        res[name] = {"envs_restarted": fresh, "us": statistics.median(events_ms(fn, reps) for _ in range(5)) * 1e3}
    del vec, bank, env
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--rounds", type=int, default=9)
    ap.add_argument("--steps", type=int, default=192)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    import marl_sat_b200 as M
    result = {"card": card(), "torch": torch.__version__, "cuda_runtime": torch.version.cuda, "rounds": args.rounds}
    print(json.dumps(result), flush=True)
    cases = (("uf100-430 x 65536 (headline)", 100, 430, 65536, (1, 0)),
             ("uf100-430 x 65536, shard 0 of 8 (8192 envs)", 100, 430, 65536, (8, 0)),
             ("uf250-1065 x 16384", 250, 1065, 16384, (1, 0)))
    result["call"] = []
    for case in cases[:2]:
        r = call_alone(M, *case)
        result["call"].append(r)
        print(json.dumps(r), flush=True)
    result["step"] = []
    for case in cases:
        res = step_cost(M, *case, args.rounds, args.steps)
        result["step"].append(res)
        for mode in ("eager", "graph"):
            r = res[mode]
            print(f"{res['case']:46s} {mode:5s} random {r['ms_per_step']['random']['median']:.4f} "
                  f"starts {r['ms_per_step']['starts']['median']:.4f} ms/step  "
                  f"overhead {1e3 * r['overhead_ms']:.1f} us ({100 * r['overhead_frac']:.1f} %)  "
                  f"spread {1e3 * r['random_spread_ms']:.1f} / {1e3 * r['starts_spread_ms']:.1f} us", flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    return 0


if __name__ == "__main__":
    sys.exit(main())
