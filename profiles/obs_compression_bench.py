"""Rollout steps into compressible versus ordinary observation memory.

Observation buffers come from ``marl_sat_b200.env.obs_empty``: compressible device memory (``msat_obs_alloc``,
CU_MEM_ALLOCATION_COMP_GENERIC) where the driver grants it.  This script measures what that memory buys.

Per workload, one ``VecSATEnv`` at ``bench.py``'s shape, seeds and de-phasing runs the launch mode ``bench.py``
picks for it (single ``msat_rollout_step`` launches, a replayed CUDA graph of 32 steps, or ``msat_rollout_steps``
with every step's observations into ``[32, B, A, D]``).  Two observation buffers of the same shape alternate: an
ordinary ``torch.empty`` one and a compressible one.  Every round restores the env state and the rng chain, so both
arms compute the same steps; the order of the arms alternates between rounds.  Reported per arm: the median,
minimum and maximum ms per step over the rounds (CUDA events), and whether the observations of the two arms are
bit-identical after the last round.

Write-only ceilings: ``fill_(-1)`` and ``zero_()`` on a buffer of the headline's observation size (4.13 GB) in
either kind of memory, median of 10.

    python profiles/obs_compression_bench.py [--rounds 9] [--steps 200] [--out result.json]
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

# the five bench.py workloads at their default sizes, then the extra shapes
WORKLOADS = {
    "uf20-91": dict(n=20, m=91, k=3, vpa=None, envs=16, kind="uniform"),
    "uf50-218": dict(n=50, m=218, k=3, vpa=None, envs=4096, kind="uniform"),
    "uf100-430": dict(n=100, m=430, k=3, vpa=None, envs=65536, kind="uniform"),
    "uf250-1065": dict(n=250, m=1065, k=3, vpa=None, envs=16384, kind="uniform"),
    "mixed-k3-7": dict(n=100, m=430, k=7, vpa=7, envs=32768, kind="mixed"),
}
CASES = [  # label, workload, global envs, (world, rank) shard, obs dtype
    ("uf100-430 x 65536 (headline)", "uf100-430", 65536, (1, 0), torch.int32),
    ("uf20-91 x 16", "uf20-91", 16, (1, 0), torch.int32),
    ("uf50-218 x 4096", "uf50-218", 4096, (1, 0), torch.int32),
    ("uf250-1065 x 16384", "uf250-1065", 16384, (1, 0), torch.int32),
    ("mixed-k3-7 x 32768", "mixed-k3-7", 32768, (1, 0), torch.int32),
    ("uf20-91 x 65536", "uf20-91", 65536, (1, 0), torch.int32),
    ("uf100-430 x 65536, shard 0 of 8 (8192 envs)", "uf100-430", 65536, (8, 0), torch.int32),
    ("uf100-430 x 65536, int8 observations", "uf100-430", 65536, (1, 0), torch.int8),
]
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


def run_case(M, label, wname, Bg, shard, obs_dtype, rounds, steps):
    from marl_sat_b200 import synth
    from marl_sat_b200.env import obs_empty
    w, dev = WORKLOADS[wname], torch.device("cuda", torch.cuda.current_device())
    env = M.SATEnv(w["n"], w["m"], MAX_STEPS, vars_per_agent=w["vpa"], verbose=False, device=dev, obs_dtype=obs_dtype)
    if w["kind"] == "mixed":
        problems = synth.mixed_ksat_torch(Bg, w["n"], w["m"], 3, w["k"], seed=20261018 + 2, device=dev)
    else:
        problems = synth.uniform_ksat_torch(Bg, w["n"], w["m"], w["k"], seed=20261018 + 2, device=dev)
    bank = env.make_bank(problems, validate=False)
    del problems
    vec = M.VecSATEnv(env, bank, Bg, M.prng_key(SEED), world_size=shard[0], rank=shard[1])
    B, A, V = vec.num_envs, env.num_agents, env.max_vars_per_agent
    gen = torch.Generator(device=dev).manual_seed(1234 + shard[1])
    actions = torch.randint(0, V + 1, (ACTION_CYCLE, B, A), generator=gen, device=dev, dtype=torch.int32)
    vec.reset()
    g = torch.arange(vec.env_offset, vec.env_offset + B, device=dev, dtype=torch.int64)
    vec.set_episode_steps((g % MAX_STEPS).to(torch.int32))          # bench.py's de-phasing
    obs_bytes_per_step = B * A * env.obs_dim * 4                     # bench.py's launch-mode rule (int32 bytes)
    mode = "multi" if obs_bytes_per_step <= 126e6 else ("graph" if B <= 16384 else "step")

    # one observation buffer (or multi-step output dict) per arm; the compressible one is what obs_empty returns
    arms = {}
    for arm in ("ordinary", "compressible"):
        if mode == "multi":
            out = vec.alloc_multi_step_outputs(G, emit_every_step=True)
            if arm == "ordinary":
                out["obs"] = torch.empty(out["obs"].shape, dtype=obs_dtype, device=dev)
            arms[arm] = {"out": out, "obs": out["obs"]}
        else:
            shape = (B, A, env.obs_dim)
            obs = torch.empty(shape, dtype=obs_dtype, device=dev) if arm == "ordinary" else obs_empty(shape, obs_dtype, dev)
            arms[arm] = {"obs": obs}
    state0, chain0, cur0 = vec.state.clone(), vec.keys._bufs.clone(), vec.keys._cur

    def restore():
        vec.state.copy_(state0)
        vec.keys._bufs.copy_(chain0)
        vec.keys._cur = cur0

    if mode == "graph":
        for arm in arms.values():
            vec.out["obs"] = arm["obs"]
            restore()
            for i in range(3):
                vec.step(actions[i])
            torch.cuda.synchronize()
            restore()
            arm["graph"] = torch.cuda.CUDAGraph()
            with torch.cuda.graph(arm["graph"]):
                for i in range(G):
                    vec.step(actions[i % ACTION_CYCLE])
            torch.cuda.synchronize()
    launches = steps // G if mode != "step" else steps
    run_len = launches * G if mode != "step" else steps

    def run(arm):
        a = arms[arm]
        if mode == "step":
            vec.out["obs"] = a["obs"]
            for i in range(steps):
                vec.step(actions[i % ACTION_CYCLE])
        elif mode == "graph":
            for _ in range(launches):
                a["graph"].replay()
        else:
            for r in range(launches):
                vec.steps(actions[(r % 2) * G:(r % 2) * G + G], a["out"])

    def timed(arm):
        restore()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run(arm)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / run_len

    for arm in arms:                   # warm-up: modules, clocks
        for _ in range(2):
            timed(arm)
    ms = {arm: [] for arm in arms}
    for r in range(rounds):
        for arm in (("ordinary", "compressible") if r % 2 == 0 else ("compressible", "ordinary")):
            ms[arm].append(timed(arm))
    identical = torch.equal(arms["ordinary"]["obs"], arms["compressible"]["obs"])
    res = {"case": label, "workload": wname, "envs_global": Bg, "envs_this_gpu": B, "shard": list(shard),
           "obs_dtype": str(obs_dtype).replace("torch.", ""), "launch_mode": mode, "steps_per_round": run_len,
           "obs_bytes_per_step": B * A * env.obs_dim * arms["ordinary"]["obs"].element_size(),
           "ms_per_step": {arm: summary(v) for arm, v in ms.items()}, "obs_bit_identical": bool(identical)}
    o, c = res["ms_per_step"]["ordinary"], res["ms_per_step"]["compressible"]
    spread = max(o["max"] - o["min"], c["max"] - c["min"])
    res["speedup_median"] = o["median"] / c["median"]
    res["gain_over_spread"] = (o["median"] - c["median"]) / spread if spread > 0 else None
    del arms, vec, bank, env
    torch.cuda.empty_cache()
    return res


def ceilings(reps=10):
    from marl_sat_b200.env import obs_empty
    dev = torch.device("cuda", torch.cuda.current_device())
    n = 65536 * 25 * 630                                # the headline's int32 observations, 4.13 GB
    out = {"bytes": 4 * n}
    for arm in ("ordinary", "compressible"):
        buf = torch.empty(n, dtype=torch.int32, device=dev) if arm == "ordinary" else obs_empty((n,), torch.int32, dev)
        for name, op in (("fill_-1", lambda: buf.fill_(-1)), ("zero_", lambda: buf.zero_())):
            op()
            torch.cuda.synchronize()
            ts = []
            for _ in range(reps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                op()
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
            med = statistics.median(ts)
            out[f"{arm} {name}"] = {"ms_median": med, "ms_min": min(ts), "ms_max": max(ts),
                                    "logical_gbs": 4 * n / (med * 1e-3) / 1e9}
        del buf
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--rounds", type=int, default=9)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--only-headline", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    import ctypes as C

    import marl_sat_b200 as M
    from marl_sat_b200 import _lib
    granted = C.c_int(0)
    _lib.check(_lib.load().msat_obs_compression(torch.cuda.current_device(), C.byref(granted)), "msat_obs_compression")
    result = {"card": card(), "compression_granted": bool(granted.value), "torch": torch.__version__,
              "cuda_runtime": torch.version.cuda, "rounds": args.rounds, "ceilings": ceilings(), "cases": []}
    print(json.dumps({k: result[k] for k in ("card", "compression_granted", "ceilings")}, indent=1), flush=True)
    for case in CASES[:1] if args.only_headline else CASES:
        res = run_case(M, *case, args.rounds, args.steps)
        result["cases"].append(res)
        o, c = res["ms_per_step"]["ordinary"], res["ms_per_step"]["compressible"]
        print(f"{res['case']:48s} {res['launch_mode']:5s} ordinary {o['median']:.4f} [{o['min']:.4f}, {o['max']:.4f}]"
              f"  compressible {c['median']:.4f} [{c['min']:.4f}, {c['max']:.4f}] ms/step  x{res['speedup_median']:.3f}"
              f"  identical={res['obs_bit_identical']}", flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    return 0 if all(c["obs_bit_identical"] for c in result["cases"]) else 1


if __name__ == "__main__":
    sys.exit(main())
