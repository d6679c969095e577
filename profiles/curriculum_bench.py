"""Cost of the curriculum primitives: the weighted auto-reset step, the weighted key derivation and the per-problem
statistics.

1. Step cost.  One ``VecSATEnv`` at ``bench.py``'s headline shape (uf100-430, 65,536 envs, 512-step episodes,
   de-phased) and on its first 8,192-env shard alternates two arms from the same saved state: the fused uniform step
   (one ``msat_rollout_step`` launch) and the weighted step (``msat_rng_chain`` -> ``msat_env_keys_weighted`` ->
   ``msat_step``), each eager (one Python call per step) and as a replayed CUDA graph of 32 steps.  The weights are
   heavy-tailed over the bank.  Median / min / max ms per step over the rounds (CUDA events); the arm order alternates.
2. ``msat_env_keys_weighted`` alone at B = 65,536 for P = 800, 65,536 and 2^20 (``msat_env_keys`` beside it), median
   over 200 launches.
3. ``msat_problem_stats`` at T = 512 x B = 65,536, every row done, for P = 1, 800 and 65,536, reading the problem
   index through the strides of a ``RolloutBuffer``-shaped state ``[T, B, 8]`` (uf100-430: one 32-byte sector per
   row).  GB/s counts the done flags, one 32-byte state sector, the solved flag and num_unsatisfied per done row and
   episode_step per solved row.

    python profiles/curriculum_bench.py [--rounds 9] [--steps 192] [--out result.json]
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

MAX_STEPS, SEED, ACTION_CYCLE, G = 512, 42, 64, 32


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


def step_cost(M, label, Bg, shard, rounds, steps):
    from marl_sat_b200 import synth
    dev = torch.device("cuda", torch.cuda.current_device())
    n, m = 100, 430
    env = M.SATEnv(n, m, MAX_STEPS, verbose=False, device=dev)
    bank = env.make_bank(synth.uniform_ksat_torch(Bg, n, m, 3, seed=20261018 + 2, device=dev), validate=False)
    vec = M.VecSATEnv(env, bank, Bg, M.prng_key(SEED), world_size=shard[0], rank=shard[1])
    B, A, V = vec.num_envs, env.num_agents, env.max_vars_per_agent
    gen = torch.Generator(device=dev).manual_seed(1234 + shard[1])
    actions = torch.randint(0, V + 1, (ACTION_CYCLE, B, A), generator=gen, device=dev, dtype=torch.int32)
    weights = torch.empty(bank.num_problems, dtype=torch.float64).exponential_(generator=torch.Generator().manual_seed(7)) ** 4
    vec.reset()
    g = torch.arange(vec.env_offset, vec.env_offset + B, device=dev, dtype=torch.int64)
    vec.set_episode_steps((g % MAX_STEPS).to(torch.int32))          # bench.py's de-phasing
    state0, chain0, cur0 = vec.state.clone(), vec.keys._bufs.clone(), vec.keys._cur

    def restore():
        vec.state.copy_(state0)
        vec.keys._bufs.copy_(chain0)
        vec.keys._cur = cur0

    def arm_weights(arm):
        vec.set_problem_weights(weights if arm == "weighted" else None)

    graphs = {}
    for arm in ("uniform", "weighted"):
        arm_weights(arm)
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
    res = {"case": label, "envs_global": Bg, "envs_this_gpu": B, "shard": list(shard), "bank_problems": bank.num_problems}
    for mode in ("eager", "graph"):
        def run(arm):
            arm_weights(arm)
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

        for arm in ("uniform", "weighted"):
            run(arm)
        ms = {"uniform": [], "weighted": []}
        for r in range(rounds):
            for arm in (("uniform", "weighted") if r % 2 == 0 else ("weighted", "uniform")):
                ms[arm].append(run(arm))
        u, w = summary(ms["uniform"]), summary(ms["weighted"])
        res[mode] = {"ms_per_step": {"uniform": u, "weighted": w},
                     "overhead_ms": w["median"] - u["median"], "overhead_frac": w["median"] / u["median"] - 1.0,
                     "uniform_spread_ms": u["max"] - u["min"]}
    vec.set_problem_weights(None)
    del graphs, vec, bank, env
    torch.cuda.empty_cache()
    return res


def env_keys(M, reps=200):
    dev = torch.device("cuda", torch.cuda.current_device())
    B = 65536
    pk = M.env.as_u32_tensor(M.prng_key(5), dev)
    idx = torch.empty(B, dtype=torch.int32, device=dev)
    keys = torch.empty((B, 2), dtype=torch.int32, device=dev)
    out = []
    for P in (800, 65536, 1 << 20):
        w = torch.empty(P, dtype=torch.float64).exponential_(generator=torch.Generator().manual_seed(P)) ** 4
        cum = torch.cumsum(M.problem_weights(w), 0).to(dev)
        row = {"P": P, "B": B}
        for name, c in (("uniform_env_keys", None), ("weighted_env_keys", cum)):
            fn = lambda: M.derive_env_keys(pk, pk, B, 0, B, P, idx, keys, c)
            for _ in range(10):
                fn()
            row[name + "_us"] = statistics.median(events_ms(fn, reps) for _ in range(5)) * 1e3
        out.append(row)
    return out


def problem_stats(M, reps=20):
    dev = torch.device("cuda", torch.cuda.current_device())
    T, B, W = 512, 65536, 8
    gen = torch.Generator(device=dev).manual_seed(3)
    state = torch.randint(0, 2 ** 31 - 1, (T, B, W), generator=gen, device=dev, dtype=torch.int32)
    done = torch.ones((T, B), dtype=torch.uint8, device=dev)
    solved = torch.randint(0, 2, (T, B), generator=gen, device=dev, dtype=torch.int32).to(torch.uint8)
    nu = torch.randint(0, 40, (T, B), generator=gen, device=dev, dtype=torch.int32) * (1 - solved.int())
    es = torch.randint(1, 512, (T, B), generator=gen, device=dev, dtype=torch.int32)
    n_done, n_solved = T * B, int(solved.sum())
    nbytes = T * B + n_done * (32 + 1 + 4) + n_solved * 4
    out = []
    for P in (1, 800, 65536):
        state[:, :, 5] = torch.randint(0, P, (T, B), generator=gen, device=dev, dtype=torch.int32)
        pidx = state[:, :, 5]
        stats = torch.zeros((P, 4), dtype=torch.int64, device=dev)
        fn = lambda: M.problem_stats(pidx, done, solved, nu, es, P, stats=stats)
        for _ in range(3):
            fn()
        ms = statistics.median(events_ms(fn, reps) for _ in range(5))
        stats.zero_()
        fn()
        ok = int(stats[:, 0].sum()) == n_done and int(stats[:, 1].sum()) == n_solved
        out.append({"P": P, "T": T, "B": B, "rows_done": n_done, "ms": ms, "bytes_read": nbytes,
                    "gbs": nbytes / (ms * 1e-3) / 1e9, "totals_ok": ok})
    p1 = next(r for r in out if r["P"] == 1)["ms"]
    pbig = next(r for r in out if r["P"] == 65536)["ms"]
    return {"cases": out, "p1_over_p65536": p1 / pbig}


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
    result["env_keys"] = env_keys(M)
    print(json.dumps(result["env_keys"]), flush=True)
    result["problem_stats"] = problem_stats(M)
    print(json.dumps(result["problem_stats"]), flush=True)
    result["step"] = []
    for case in (("uf100-430 x 65536 (headline)", 65536, (1, 0)), ("uf100-430 x 65536, shard 0 of 8 (8192 envs)", 65536, (8, 0))):
        res = step_cost(M, *case, args.rounds, args.steps)
        result["step"].append(res)
        for mode in ("eager", "graph"):
            r = res[mode]
            print(f"{res['case']:46s} {mode:5s} uniform {r['ms_per_step']['uniform']['median']:.4f} "
                  f"weighted {r['ms_per_step']['weighted']['median']:.4f} ms/step  "
                  f"overhead {1e3 * r['overhead_ms']:.1f} us ({100 * r['overhead_frac']:.1f} %)", flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    return 0 if all(c["totals_ok"] for c in result["problem_stats"]["cases"]) else 1


if __name__ == "__main__":
    sys.exit(main())
