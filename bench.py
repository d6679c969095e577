#!/usr/bin/env python
"""Benchmark of the batched SATEnv hot path (BASELINE.json metric: SATEnv env-steps/s, uf100-430).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

One "step" = one rollout step of every environment: the device RNG chain (learner:397-434), the
per-env problem-index / reset-key derivation and the fused flip + clause evaluation + reward / done /
info + auto-reset + observation kernel.  The global batch (65,536 envs for the headline workload) is
sharded across the N ranks in contiguous blocks with no collective on the step path; `value` is
global env-steps/s from CUDA-event time, max over ranks.  Rank 0 prints ONE JSON line.

`--impl reference` times the CPU restatement of the reference algorithm (oracle/: plain C + OpenMP on all
host cores; NumPy, one process per core, if gcc is missing) on a bounded sample of the same workload: the reference's own JAX build cannot run here
(no JAX in the image), see DESIGN.md section 6.
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import os
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (it may be read-only)

METRIC = "SATEnv env-steps/s, uf100-430, 1/2/4/8 B200; achieved HBM GB/s vs peak"
UNIT = "env-steps/s"

# name -> shape (BASELINE.json configs / SURVEY.md Appendix C)
WORKLOADS = {
    "uf20-91": dict(n=20, m=91, k=3, vpa=None, envs=16, kind="uniform"),
    "uf50-218": dict(n=50, m=218, k=3, vpa=None, envs=4096, kind="uniform"),
    "uf100-430": dict(n=100, m=430, k=3, vpa=None, envs=65536, kind="uniform"),      # headline
    "uf250-1065": dict(n=250, m=1065, k=3, vpa=None, envs=16384, kind="uniform"),
    "mixed-k3-7": dict(n=100, m=430, k=7, vpa=7, envs=32768, kind="mixed"),
}
MAX_STEPS = 512          # configs/MAPPO_CONFIG.yaml:14
SEED = 42                # configs/MAPPO_CONFIG.yaml:6
ACTION_CYCLE = 64        # pre-generated action batches, cycled
DUMP_BYTES = 60 * 10**6  # --dump-outputs: array bytes written, under 64 MB with the .npy headers


def _load_synth():
    spec = importlib.util.spec_from_file_location("_msat_synth", ROOT / "marl_sat_b200" / "synth.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def make_formulas(w, count, seed):
    synth = _load_synth()
    if w["kind"] == "mixed":
        return synth.mixed_ksat(count, w["n"], w["m"], 3, w["k"], seed)
    return synth.uniform_ksat(count, w["n"], w["m"], w["k"], seed)


def algorithmic_bytes_per_env_step(n, m, k, A):
    """SURVEY.md section 8(d): obs write + literals read + packed state r/w + actions + rewards +
    dones + info + reset key / problem index."""
    D = 2 * n + m
    return (4 * A * D + 4 * m * k + 2 * (4 * ((n + 31) // 32) + 4 * ((m + 31) // 32) + 8)
            + 4 * A + 4 * A + (A + 1) + 9 + 12)


# ----------------------------------------------------------------------------------------------
# CPU restatement arm (oracle/): one process per core, each stepping its own shard of envs
# ----------------------------------------------------------------------------------------------
def _cpu_worker(args):
    wname, envs, steps, warmup, seed = args
    import numpy as np
    from oracle import rollout as orollout
    from oracle import threefry as otf
    from oracle.sat_env import SATEnvOracle
    w = WORKLOADS[wname]
    problems = make_formulas(w, envs, seed)
    env = SATEnvOracle(w["n"], w["m"], MAX_STEPS, vars_per_agent=w["vpa"])
    key, idx, rk = orollout.initial_reset_inputs(otf.prng_key(seed), envs, envs)
    _, st = env.reset(problems[idx], rk)
    rng = np.random.default_rng(seed)
    t0 = 0.0
    for i in range(warmup + steps):
        if i == warmup:
            t0 = time.perf_counter()
        acts = rng.integers(0, env.max_vars_per_agent + 1, size=(envs, env.num_agents)).astype(np.int32)
        ks = orollout.rollout_keys(key, envs, envs)
        key = ks["rng"]
        _, st, _, _, _ = orollout.env_step_with_autoreset(env, st, acts, problems, ks["new_problem_indices"],
                                                          ks["reset_keys"])
    return time.perf_counter() - t0


def run_cpu_restatement_c(wname, envs_per_core, steps, warmup, total_envs=None):
    """Compiled CPU baseline: the plain-C + OpenMP restatement (oracle/sat_env_c.c), all host cores."""
    import numpy as np
    from oracle import rollout as orollout
    from oracle import threefry as otf
    from oracle.c_port import SATEnvOracleC
    w = WORKLOADS[wname]
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    env = SATEnvOracleC(w["n"], w["m"], MAX_STEPS, vars_per_agent=w["vpa"])
    env.set_threads(cores)              # torchrun exports OMP_NUM_THREADS=1 to every rank
    threads = env.num_threads()
    envs = total_envs or envs_per_core * max(cores, 1)
    problems = make_formulas(w, envs, 1000)
    key, idx, rk = orollout.initial_reset_inputs(otf.prng_key(SEED), envs, envs)
    st = env.reset(problems[idx], rk)
    rng = np.random.default_rng(0)
    acts = [rng.integers(0, env.V + 1, size=(envs, env.A)).astype(np.int32) for _ in range(4)]
    t0 = 0.0
    for i in range(warmup + steps):
        if i == warmup:
            t0 = time.perf_counter()
        chain, nidx, keys = env.rollout_keys(key, envs, envs)
        key = chain[:2].copy()
        env.step(st, acts[i % 4], problems, nidx, keys)
    t = time.perf_counter() - t0
    return {"value": envs * steps / t, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{wname}: {envs} envs x {steps} steps (+{warmup} warm-up) of the plain-C/OpenMP restatement "
                      f"(oracle/sat_env_c.c: step all, reset all, select by done; learner:418-464) on {threads} "
                      f"threads, {t:.2f} s"}, t


def run_cpu_restatement(wname, envs_per_worker, steps, warmup):
    try:
        return run_cpu_restatement_c(wname, envs_per_worker, steps, warmup)
    except Exception as e:      # no gcc / OpenMP: fall back to the NumPy restatement, one process per core
        print(f"[bench] C restatement unavailable ({e!r}); timing the NumPy one", file=sys.stderr)
    import multiprocessing as mp
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    ctx = mp.get_context("spawn")       # safe next to an initialised CUDA context; workers import NumPy only
    jobs = [(wname, envs_per_worker, steps, warmup, 1000 + i) for i in range(cores)]
    with ctx.Pool(cores) as pool:
        times = pool.map(_cpu_worker, jobs)
    t = max(times)
    total = envs_per_worker * cores * steps
    return {"value": total / t, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{wname}: {cores} processes x {envs_per_worker} envs x {steps} steps (+{warmup} warm-up) of the "
                      f"NumPy restatement (step all, reset all, select by done; learner:418-464), "
                      f"{t:.2f} s"}, t


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    wname = args.workload
    w = WORKLOADS[wname]
    envs_per_worker = args.cpu_envs_per_core
    base, t = run_cpu_restatement(wname, envs_per_worker, args.steps, args.warmup)
    cores = base["cores"]
    line = {
        "impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / max(1, args.steps),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": f"{wname} (n={w['n']}, m={w['m']}, k={w['k']}), bounded sample per step on "
                               f"{cores} host threads: {base['sample']}",
                   "max_steps": MAX_STEPS, "auto_reset": True},
        "cpu_baseline": base,
        "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "CPU restatement of the reference algorithm (oracle/: plain C + OpenMP, NumPy fallback); the "
                "reference's JAX build is not installable in this image (no jax wheel, no network)",
    }
    print(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------------------------
# clocks (NVML sampled in a thread during the timed region)
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, torch_device_index):
        self.samples = []
        self._stop = threading.Event()
        self._thread = None
        self.max_mhz = None
        self.ok = False
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(torch_device_index).uuid)
            if not uuid.startswith("GPU-"):
                uuid = "GPU-" + uuid
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(torch_device_index)
            self.nv = pynvml
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:          # pragma: no cover
            self.err = repr(e)
            self._init_smi(torch_device_index)

    # fallback when NVML's Python binding is unusable: poll nvidia-smi (the recipe's clocks line)
    def _init_smi(self, index):     # pragma: no cover
        import shutil
        import subprocess
        if not shutil.which("nvidia-smi"):
            return
        try:
            import torch
            uuid = str(torch.cuda.get_device_properties(index).uuid)
            sel = uuid if uuid.startswith("GPU-") else "GPU-" + uuid
            q = subprocess.run(["nvidia-smi", "-i", sel, "--query-gpu=clocks.max.sm", "--format=csv,noheader,nounits"],
                               capture_output=True, text=True, timeout=20)
            self.max_mhz = int(q.stdout.strip().splitlines()[0])
            self._smi = subprocess.Popen(
                ["nvidia-smi", "-i", sel, "--query-gpu=clocks.sm,clocks_event_reasons.active",
                 "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.nv = None
            self.ok = True
        except Exception as e:
            self.err += " / nvidia-smi: " + repr(e)

    def _loop_smi(self):            # pragma: no cover
        for line in self._smi.stdout:
            if self._stop.is_set():
                break
            try:
                mhz, reasons = [x.strip() for x in line.split(",")[:2]]
                self.samples.append((time.perf_counter(), int(mhz), int(reasons, 16)))
            except Exception:
                pass

    def _loop(self):
        if self.nv is None:
            return self._loop_smi()
        nv = self.nv
        while not self._stop.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((time.perf_counter(), mhz, reasons))
            except Exception:
                pass
            time.sleep(0.010)

    def start(self):
        if self.ok:
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()

    def stop(self):
        if self._thread:
            self._stop.set()
            if getattr(self, "_smi", None) is not None:
                self._smi.terminate()
            self._thread.join(timeout=2)

    def summary(self, t0, t1):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "error": getattr(self, "err", "nvml unavailable")}
        inside = [s for s in self.samples if t0 <= s[0] <= t1]
        window = "timed region"
        if len(inside) < 3:
            inside, window = self.samples, "whole loaded period (timed region too short to sample)"
        mhz = sorted(s[1] for s in inside)
        bits = 0
        for s in inside:
            bits |= s[2]
        return {"sm_mhz": mhz[len(mhz) // 2] if mhz else None, "sm_max_mhz": self.max_mhz,
                "reasons": [name for bit, name in self.REASONS.items() if bits & bit],
                "samples": len(inside), "window": window}


# ----------------------------------------------------------------------------------------------
# CUDA arm
# ----------------------------------------------------------------------------------------------
def _time_steps(torch, fn, count):
    """CUDA-event time (ms) of `count` calls of fn(i) on the current stream."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(count):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def dump_step_outputs(out, directory, row=None):
    """Write the arrays one rollout step returned -- ``out`` of ``VecSATEnv.step``, or row ``row`` of the
    ``[K, B, ...]`` outputs of ``VecSATEnv.steps`` -- as ``directory/<name>.npy`` in float32 (every value is
    float32 or a small integer, so the cast is exact).  When they exceed DUMP_BYTES together, the same fixed,
    seeded sample of env rows is taken from each; ``env_index.npy`` lists the rows written."""
    import numpy as np
    import torch
    arrays = {k: (v if row is None else v[row]) for k, v in out.items()     # "_block": storage behind the views
              if isinstance(v, torch.Tensor) and not k.startswith("_")}
    B = arrays["reward"].shape[0]
    bytes_per_env = sum(4 * a[0].numel() for a in arrays.values()) + 8
    rows = np.arange(B)
    if bytes_per_env * B > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(B, DUMP_BYTES // bytes_per_env, replace=False))
    idx = torch.from_numpy(rows).to(arrays["reward"].device)
    directory = Path(directory)
    directory.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(directory / f"{name}.npy", a.index_select(0, idx).float().cpu().numpy())
    np.save(directory / "env_index.npy", rows.astype(np.float64))


def main_ours(args):
    import torch
    import torch.distributed as dist

    import marl_sat_b200 as M

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if args.gpus != world and rank == 0:
        print(f"[bench] note: --gpus {args.gpus} but WORLD_SIZE={world}; using {world}", file=sys.stderr)

    wname = args.workload
    w = WORKLOADS[wname]
    Bg = args.envs or w["envs"]
    if args.scaling == "weak":
        Bg *= world
    # debugging aid: run the shard that rank R of an N-rank job would own, alone on this GPU
    shard_world, shard_rank = (args.emulate_shard if args.emulate_shard else (world, rank))
    env = M.SATEnv(w["n"], w["m"], MAX_STEPS, vars_per_agent=w["vpa"], verbose=False, device=dev,
                   group_threads=args.group_threads)
    P = args.problems or Bg
    # synthetic formulas are drawn on the device (same distribution as the NumPy generator the tests use)
    from marl_sat_b200 import synth
    if w["kind"] == "mixed":
        problems = synth.mixed_ksat_torch(P, w["n"], w["m"], 3, w["k"], seed=20261018 + 2, device=dev)
    else:
        problems = synth.uniform_ksat_torch(P, w["n"], w["m"], w["k"], seed=20261018 + 2, device=dev)
    bank = env.make_bank(problems, validate=False)
    del problems
    vec = M.VecSATEnv(env, bank, Bg, M.prng_key(SEED), world_size=shard_world, rank=shard_rank)
    B = vec.num_envs
    A, V = env.num_agents, env.max_vars_per_agent
    gen = torch.Generator(device=dev).manual_seed(1234 + shard_rank)
    actions = torch.randint(0, V + 1, (ACTION_CYCLE, B, A), generator=gen, device=dev, dtype=torch.int32)

    def dephase(v):
        """Fresh batch -> steady state: env g starts at episode step g mod max_steps, so ~B/max_steps envs time
        out (and auto-reset inside the step kernel) at EVERY rollout step instead of all of them at step 512."""
        g = torch.arange(v.env_offset, v.env_offset + v.num_envs, device=dev, dtype=torch.int64)
        v.set_episode_steps((g % v.env.max_steps).to(torch.int32))

    vec.reset()
    dephase(vec)
    reset_counter = torch.zeros(1, dtype=torch.int64, device=dev)
    env.count_resets(w["k"], reset_counter)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()

    K, W = args.steps, args.warmup
    # e2e leg: same envs API with compact outputs (one reward / done value per env: every agent's is the same
    # scalar, env:196,260, and the host side re-expands them as views); it shares the observation buffer.
    # Pinned host buffers are allocated up front (no allocation between timed regions).
    vec_h = M.VecSATEnv(env, bank, Bg, M.prng_key(SEED + 1), world_size=shard_world, rank=shard_rank, emit_obs=False,
                        compact_outputs=True)
    vec_h.out["obs"] = vec.out["obs"]
    vec_h.reset()
    dephase(vec_h)
    host = vec_h.alloc_host_io()
    slots = vec_h.alloc_async_io(depth=2)
    host_actions = [actions[i].cpu().pin_memory() for i in range(4)]
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()

    # ---- device-resident throughput: `value` -------------------------------------------------
    # bring the GPU to its steady clocks first (>= 60 ms of steps), then the W warm-up steps the caller asked for.
    # The clock warm-up runs as many steps as fit its wall-clock window, so the env state and the rng chain are
    # put back afterwards (in place: the step binds their addresses): what the timed steps compute depends on
    # the arguments alone.
    state0, chain0, cur0 = vec.state.clone(), vec.keys._bufs.clone(), vec.keys._cur
    t_pre = time.perf_counter()
    while time.perf_counter() - t_pre < 0.06:
        for i in range(8):
            vec.step(actions[i])
        torch.cuda.synchronize()
    vec.state.copy_(state0)
    vec.keys._bufs.copy_(chain0)
    vec.keys._cur = cur0
    del state0, chain0
    for i in range(W):
        vec.step(actions[i % ACTION_CYCLE])
    torch.cuda.synchronize()
    graph = None
    obs_bytes_per_step = B * A * env.obs_dim * 4
    mode = args.launch
    if mode == "auto":
        # L2-resident batches are launch/latency-bound: K fused steps per launch; up to 16,384 envs per GPU the
        # ~85-170 us step is short enough for the launch gap to show: CUDA graphs; above that plain launches
        mode = "multi" if obs_bytes_per_step <= 126e6 else ("graph" if B <= 16384 else "step")
    if args.graph >= 0:
        mode = "graph" if args.graph > 0 else ("step" if mode == "graph" else mode)
    G = 0
    multi_out = None
    if mode == "graph":
        # capture a block of G rollout steps (G even, so the ping-pong rng buffers end where they started) and
        # replay it; the remainder is launched directly
        G = max(2, (args.graph if args.graph > 0 else 32) // 2 * 2)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for i in range(G):
                vec.step(actions[i % ACTION_CYCLE])
        torch.cuda.synchronize()
    elif mode == "multi":
        # msat_rollout_steps: 32 steps of the pre-generated action table per launch, the int32 observations of
        # EVERY step written to a [32, B, A, D] buffer (same bytes per step as the single-step launch)
        G = 32
        multi_out = vec.alloc_multi_step_outputs(G, emit_every_step=True)
        vec.steps(actions[:G], multi_out)
        torch.cuda.synchronize()

    def run_steps(count, first):
        if mode == "step":
            for i in range(count):
                vec.step(actions[(first + i) % ACTION_CYCLE])
            return
        reps, rem = divmod(count, G)
        if mode == "graph":
            for _ in range(reps):
                graph.replay()
            for i in range(rem):
                vec.step(actions[i % ACTION_CYCLE])
        else:
            for r in range(reps):
                vec.steps(actions[(r % 2) * G:(r % 2) * G + G], multi_out)
            if rem:
                vec.steps(actions[:rem], multi_out)

    barrier()
    reset_counter.zero_()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.perf_counter()
    ev0.record()
    run_steps(K, W)
    ev1.record()
    torch.cuda.synchronize()
    t_wall1 = time.perf_counter()
    if sampler:
        sampler.stop()
    barrier()
    ms = ev0.elapsed_time(ev1)
    resets_timed = int(reset_counter.item())
    if args.dump_outputs and rank == 0:
        if mode == "multi":         # the last launch wrote rows 0 .. (K mod G or G) - 1
            dump_step_outputs(multi_out, args.dump_outputs, row=(K % G or G) - 1)
        else:
            dump_step_outputs(vec.out, args.dump_outputs)
    launches = K if mode != "multi" else (K // G + (1 if K % G else 0))    # fused step launches in the timed region

    # ---- dominant kernel alone (roofline): K launches of the same fused step, back to back ---------------
    for i in range(3):
        vec.step(actions[i])
    torch.cuda.synchronize()
    kernel_ms = _time_steps(torch, lambda i: vec.step(actions[i % ACTION_CYCLE]), K) / K

    # ---- auto-reset cost: the same step with 25 % and 100 % of the envs resetting every step -----------------
    reset_legs = {}
    if not args.no_reset_legs:
        for label, max_steps in (("reset_heavy", 4), ("all_reset", 1)):
            env_r = M.SATEnv(w["n"], w["m"], max_steps, vars_per_agent=w["vpa"], verbose=False, device=dev,
                             group_threads=args.group_threads)
            vec_r = M.VecSATEnv(env_r, bank.for_env(env_r), Bg, M.prng_key(SEED + 3), world_size=shard_world,
                                rank=shard_rank, emit_obs=False)
            vec_r.out["obs"] = vec.out["obs"]
            cnt = torch.zeros(1, dtype=torch.int64, device=dev)
            env_r.count_resets(w["k"], cnt)
            vec_r.reset()
            dephase(vec_r)
            for i in range(4):
                vec_r.step(actions[i])
            cnt.zero_()
            Kr = min(K, 40)
            r_ms = _time_steps(torch, lambda i: vec_r.step(actions[i % ACTION_CYCLE]), Kr) / Kr
            reset_legs[label] = {"max_steps": max_steps, "ms_per_step": r_ms, "steps": Kr,
                                 "autoreset_frac": int(cnt.item()) / float(B * Kr),
                                 "value": Bg / (r_ms * 1e-3)}
            env_r.count_resets(w["k"], None)
            del vec_r, env_r

    # ---- end to end through the host-buffer entry points: `e2e` ------------------------------------------------
    # Double-buffered pipeline (msat_rollout_step_host_async): per step the host hands over a pinned action
    # batch, the library uploads it, runs the fused step and downloads reward / done / info into pinned
    # memory; the host reads the results of step t-2 while steps t-1 and t are in flight.
    Ke = max(4, min(K, args.e2e_steps))
    sink = [0]

    def harvest(slot):
        vec_h.host_wait(slot)
        h = slots[slot]["host"]
        sink[0] += int(h["solved"][0]) + int(h["done"][0, 0])     # the host reads the step's result

    def e2e_async(n):
        for t in range(n):
            sl = t & 1
            if t >= 2:
                harvest(sl)
            vec_h.step_host_async(sl, slots[sl], actions_host=host_actions[t % 4])
        harvest(n & 1)
        harvest((n + 1) & 1)
    e2e_async(4)
    torch.cuda.synchronize()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tw0 = time.perf_counter()
    e0.record()
    e2e_async(Ke)
    e1.record()
    torch.cuda.synchronize()
    e2e_wall_ms = 1e3 * (time.perf_counter() - tw0)
    barrier()
    e2e_ms = max(e0.elapsed_time(e1), 0.0)
    # the synchronous single-call variant (msat_rollout_step_host: upload, step, download, stream sync per call)
    for i in range(2):
        host["actions"] = host_actions[i % 4]
        vec_h.step_host(host)
    torch.cuda.synchronize()
    barrier()

    def sync_step(i):
        host["actions"] = host_actions[i % 4]
        vec_h.step_host(host)
        rewards, dones, infos = vec_h.host_views(host)      # reference-shaped dicts (views)
        sink[0] += int(infos["solved"][0]) + int(dones["__all__"][0])
    Ks = min(Ke, 30)
    e2e_sync_ms = _time_steps(torch, sync_step, Ks)
    barrier()
    h2d = B * A * 4
    d2h = B * (4 + 1 + 1 + 4 + 4)           # team reward, done, solved, num_unsatisfied, episode_step

    # optional: also bring the observations to the host (PCIe-bound; reported separately)
    e2e_obs = None
    if args.e2e_obs_steps > 0 and world == 1:
        obs_host = torch.empty(vec.out["obs"].shape, dtype=torch.int32, pin_memory=True)
        o0, o1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        vec_h.step_host(host)
        obs_host.copy_(vec.out["obs"], non_blocking=True)
        torch.cuda.synchronize()
        barrier()
        o0.record()
        for i in range(args.e2e_obs_steps):
            vec_h.step_host(host)
            obs_host.copy_(vec.out["obs"], non_blocking=True)
            torch.cuda.synchronize()
        o1.record()
        torch.cuda.synchronize()
        e2e_obs = (o0.elapsed_time(o1), obs_host.numel() * 4)
        del obs_host

    # ---- K fused steps per launch (msat_rollout_steps): launch-bound small batches -----------------------------
    kstep_info = None
    if not args.no_kstep_leg and B <= 16384:
        Kf = 32
        outs = vec.alloc_multi_step_outputs(Kf, emit_every_step=False)
        outs["obs"] = vec.out["obs"]
        tbl = actions[:Kf].contiguous()
        for _ in range(2):
            vec.steps(tbl, outs)
        reps = max(1, min(K, 320) // Kf)
        f_ms = _time_steps(torch, lambda i: vec.steps(tbl, outs), reps) / (reps * Kf)
        del outs
        obs_all = None
        try:
            outs_all = vec.alloc_multi_step_outputs(Kf, emit_every_step=True)
            for _ in range(2):
                vec.steps(tbl, outs_all)
            fa_ms = _time_steps(torch, lambda i: vec.steps(tbl, outs_all), reps) / (reps * Kf)
            del outs_all
        except torch.OutOfMemoryError:
            fa_ms = None
        kstep_info = {"steps_per_launch": Kf, "launches": reps,
                      "final_obs_only": {"ms_per_step": f_ms, "value": Bg / (f_ms * 1e-3),
                                         "what": "K steps per launch, observations of the final state only"},
                      "obs_every_step": None if fa_ms is None else {
                          "ms_per_step": fa_ms, "value": Bg / (fa_ms * 1e-3),
                          "what": "K steps per launch, int32 observations written for every step into [K,B,A,D]"},
                      "what": "msat_rollout_steps: one launch for 32 rollout steps of an action table; state and "
                              "formula stay in shared memory across the steps"}

    # ---- MAPPO advantage path on the same batch (learner:504-532): T x B GAE scan + normalisation -------
    gae_info = None
    if not args.no_gae:
        T = args.gae_steps
        gg = torch.Generator(device=dev).manual_seed(7 + shard_rank)
        g_reward = (torch.rand((T, B), generator=gg, device=dev) < 0.01).float()
        g_done = (torch.rand((T, B), generator=gg, device=dev) < 0.005).to(torch.uint8)
        g_value = torch.randn((T, B), generator=gg, device=dev)
        g_last = torch.randn((B,), generator=gg, device=dev)
        adv = torch.empty((T, B), dtype=torch.float32, device=dev)
        tgt = torch.empty((T, B), dtype=torch.float32, device=dev)
        stats = torch.zeros(3, dtype=torch.float64, device=dev)
        reps = 10

        def scan_once():
            stats.zero_()
            M.calculate_gae(g_reward, g_done, g_value, g_last, 0.995, 0.95, stats=stats, out=(adv, tgt))

        gstats = [stats]

        def norm_once():
            M.normalize_advantages(adv, stats=gstats[0], reduced=True)    # the kernel alone (statistics already global)
        for _ in range(3):
            scan_once()
        raw = adv.clone()
        allreduce_us = None
        if world > 1:
            # the one collective of the advantage path: NCCL all-reduce of (count, sum, sum of squares), 24 bytes
            for _ in range(3):
                gstats[0] = M.allreduce_stats(stats)
            torch.cuda.synchronize()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(20):
                gstats[0] = M.allreduce_stats(stats)
            a1.record()
            torch.cuda.synchronize()
            allreduce_us = a0.elapsed_time(a1) * 1e3 / 20
        norm_once()
        torch.cuda.synchronize()
        g0, g1, g2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        # replayed as CUDA graphs of `reps` launches each: the ~100 us / ~40 us kernels (10-30 us on the shards of a
        # multi-GPU run) are timed without the Python wrapper's per-call work; no collective is captured (the
        # statistics all-reduce is timed separately above)
        gs_, gn_ = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        with torch.cuda.graph(gs_):
            for _ in range(reps):
                scan_once()
        with torch.cuda.graph(gn_):
            for _ in range(reps):
                norm_once()
        gs_.replay()                    # first replay uploads the graph: untimed
        gn_.replay()
        torch.cuda.synchronize()
        g0.record()
        gs_.replay()
        g1.record()
        gn_.replay()
        g2.record()
        torch.cuda.synchronize()
        scan_ms, norm_ms = g0.elapsed_time(g1) / reps, g1.elapsed_time(g2) / reps
        gae_info = {"num_steps": T, "num_envs": B, "scan_ms": scan_ms, "normalize_ms": norm_ms,
                    "scan_bytes_per_element": 17, "scan_gbs": 17.0 * T * B / (scan_ms * 1e-3) / 1e9,
                    "normalize_bytes_per_element": 8, "normalize_gbs": 8.0 * T * B / (norm_ms * 1e-3) / 1e9,
                    "note": "synthetic rollout, inputs resident in HBM; 17 B/element = reward 4 + done 1 + value 4 + "
                            "adv 4 + target 4, advantage statistics accumulated in the same pass; normalisation = "
                            "one in-place map (8 B) with already reduced statistics",
                    "stats_allreduce_us": allreduce_us}
        if world > 1 and Bg % world == 0:
            # self-check of the sharded normalisation: gather every rank's raw advantages on rank 0 and compare
            # the sharded result with the full-batch computation
            stats.zero_()
            M.calculate_gae(g_reward, g_done, g_value, g_last, 0.995, 0.95, stats=stats, out=(adv, tgt))
            raw = adv.clone()
            M.normalize_advantages(raw, stats=stats)
            parts = [torch.empty_like(g_value) for _ in range(world)] if rank == 0 else None
            raws = [torch.empty_like(g_value) for _ in range(world)] if rank == 0 else None
            adv2 = adv
            dist.gather(raw, parts, dst=0)
            dist.gather(adv2, raws, dst=0)
            if rank == 0:
                full = torch.cat(raws, dim=1).double()
                ref = (full - full.mean()) / (full.var(unbiased=False).sqrt() + 1e-8)
                err = (torch.cat(parts, dim=1).double() - ref).abs().max().item()
                gae_info["sharded_vs_full_batch_max_abs_err"] = err
                if err > 1e-4:
                    raise SystemExit(f"sharded advantage normalisation differs from the full batch: {err}")
        del g_reward, g_done, g_value, g_last, adv, tgt

    # ---- extra: the reference policy's actual input (SURVEY.md F8 / section 8f rank 1) ----------------------
    # its networks read the GNN input, never the local observations, so a GNN-style consumer can skip the
    # 63 KB/env observation write: rollout step without obs + per-step dynamic GNN features.  Reported as an
    # extra key only; the headline metric above always includes the observations.
    gnn_info = None
    if world == 1 and not args.no_gnn_leg:
        from marl_sat_b200.features import static_graph
        vec_g = M.VecSATEnv(env, bank, Bg, M.prng_key(SEED + 2), emit_obs=False, compact_outputs=True,
                            gnn_outputs=True)
        vec_g.reset()
        dephase(vec_g)
        static_graph(bank)                      # per-formula part, once
        for i in range(5):
            vec_g.step(actions[i])
        torch.cuda.synchronize()
        Kg = min(K, 100)
        g_ms = _time_steps(torch, lambda i: vec_g.step(actions[i % ACTION_CYCLE]), Kg) / Kg
        d = bank.plan.dims
        lits_bytes = (w["m"] * w["k"] * 2 + 15) // 16 * 16
        g_bytes = (4 * w["n"] + 12 * w["m"] + lits_bytes + 2 * 4 * d.state_words + 4 * A + 4 + 1 + 1 + 4 + 4)
        gnn_info = {"value": Bg / (g_ms * 1e-3), "unit": UNIT, "ms_per_step": g_ms, "steps": Kg,
                    "bytes_out_per_env_step": 4 * w["n"] + 12 * w["m"],
                    "bytes_moved_per_env_step": g_bytes,
                    "gbs": g_bytes * B / (g_ms * 1e-3) / 1e9,
                    "what": "msat_rollout_step_gnn: one launch per step, no local observations, dynamic GNN input "
                            "(assignment int32[B,n], clause_features float32[B,m,3]) emitted from the staged literal "
                            "block; static graph features emitted once per formula bank; bytes_moved = outputs + "
                            "packed literal block + state r/w + actions + reward/done/info"}
        del vec_g
        # the same launches with the incremental clause update (north_star: CSR var -> clause occurrence lists,
        # only the clauses adjacent to flipped variables are touched): its own bank (records carry the CSR) and
        # state (4-bit true-literal counts per clause); results are bit-identical (tests/test_fuzz_cuda.py)
        try:
            env_i = M.SATEnv(w["n"], w["m"], MAX_STEPS, vars_per_agent=w["vpa"], verbose=False, device=dev,
                             clause_update="incremental")
            if w["kind"] == "mixed":
                pr = synth.mixed_ksat_torch(P, w["n"], w["m"], 3, w["k"], seed=20261018 + 2, device=dev)
            else:
                pr = synth.uniform_ksat_torch(P, w["n"], w["m"], w["k"], seed=20261018 + 2, device=dev)
            bank_i = env_i.make_bank(pr, validate=False)
            del pr
            legs = {}
            # a second action distribution: a policy that mostly waits -- every agent picks the no-op action V
            # with probability 0.95, so ~1.25 of the 25 agents flip per step (uniform actions: ~20)
            noop = torch.rand((ACTION_CYCLE, B, A), generator=gen, device=dev) < 0.95
            sparse = torch.where(noop, torch.full_like(actions, V), actions)
            del noop
            for label, kw, acts in (("gnn_input", dict(gnn_outputs=True), actions), ("state_only", dict(), actions),
                                    ("gnn_input_sparse_flips", dict(gnn_outputs=True), sparse),
                                    ("state_only_sparse_flips", dict(), sparse)):
                res = {}
                for variant, (e_, b_) in (("full", (env, bank)), ("incremental", (env_i, bank_i))):
                    v = M.VecSATEnv(e_, b_, Bg, M.prng_key(SEED + 2), emit_obs=False, compact_outputs=True, **kw)
                    v.reset()
                    dephase(v)
                    for i in range(5):
                        v.step(acts[i])
                    torch.cuda.synchronize()
                    res[variant] = _time_steps(torch, lambda i: v.step(acts[i % ACTION_CYCLE]), Kg) / Kg
                    del v
                legs[label] = {"full_ms_per_step": res["full"], "incremental_ms_per_step": res["incremental"],
                               "incremental_speedup": res["full"] / res["incremental"]}
            del sparse
            di = bank_i.plan.dims
            gnn_info["clause_update_variants"] = {
                **legs, "rec_bytes": {"full": d.rec_bytes, "incremental": di.rec_bytes},
                "state_bytes": {"full": 4 * d.state_words, "incremental": 4 * di.state_words},
                "what": "gnn_input: msat_rollout_step_gnn; state_only: msat_rollout_step with obs == NULL (reward / "
                        "done / info only).  full = every clause re-evaluated from the staged literal block; "
                        "incremental = +-1 updates of the adjacent clauses' counts from the CSR rows of the flipped "
                        "variables, no literal block unless the episode restarts; *_sparse_flips = 95 % of the agents choose "
                        "the no-op action (~1.25 flips per env-step instead of ~20)"}
            del bank_i, env_i
        except torch.OutOfMemoryError:
            pass
    # ---- extra: the same step with int8 observations (MSAT_OBS_INT8): same values, a quarter of the bytes --------
    # for consumers that cast the observations anyway; the headline metric above is always the int32 contract.
    i8_info = None
    if world == 1 and not args.no_gnn_leg:
        env8 = M.SATEnv(w["n"], w["m"], MAX_STEPS, vars_per_agent=w["vpa"], verbose=False, device=dev,
                        group_threads=args.group_threads, obs_dtype=torch.int8)
        vec8 = M.VecSATEnv(env8, bank.for_env(env8), Bg, M.prng_key(SEED + 4))
        vec8.reset()
        dephase(vec8)
        for i in range(5):
            vec8.step(actions[i])
        torch.cuda.synchronize()
        K8 = min(K, 100)
        i8_ms = _time_steps(torch, lambda i: vec8.step(actions[i % ACTION_CYCLE]), K8) / K8
        d8 = bank.plan.dims
        copy_bytes = (w["m"] * w["k"] * 2 + 15) // 16 * 16 + 4 * ((A * env.obs_dim + 31) // 32 + 1)
        i8_bytes = A * env.obs_dim + copy_bytes + 2 * 4 * d8.state_words + 4 * A + 4 * A + (A + 1) + 9 + 12
        i8_info = {"value": Bg / (i8_ms * 1e-3), "unit": UNIT, "ms_per_step": i8_ms, "steps": K8,
                   "bytes_moved_per_env_step": i8_bytes, "gbs": i8_bytes * B / (i8_ms * 1e-3) / 1e9,
                   "what": "msat_rollout_step on a plan with msat_plan_set_obs_dtype(MSAT_OBS_INT8): observations "
                           "int8[B,A,D] with the same -1/0/1 values (parity: tests/test_round2_cuda.py); bytes_moved = "
                           "int8 observations + staged bank record (packed literals + agent-mask stream) + state r/w "
                           "+ actions + reward/done/info"}
        del vec8, env8
    env.count_resets(w["k"], None)

    # ---- reduce over ranks (max time) ------------------------------------------------------------------
    t = torch.tensor([ms, kernel_ms, e2e_ms, e2e_obs[0] if e2e_obs else 0.0, e2e_sync_ms, e2e_wall_ms,
                      reset_legs.get("reset_heavy", {}).get("ms_per_step", 0.0),
                      reset_legs.get("all_reset", {}).get("ms_per_step", 0.0),
                      gae_info["scan_ms"] if gae_info else 0.0, gae_info["normalize_ms"] if gae_info else 0.0],
                     dtype=torch.float64, device=dev)
    rs = torch.tensor([resets_timed], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(rs, op=dist.ReduceOp.SUM)
    (ms, kernel_ms_max, e2e_ms, e2e_obs_ms, e2e_sync_ms, e2e_wall_ms, heavy_ms, allr_ms, scan_ms_max,
     norm_ms_max) = [float(x) for x in t.tolist()]
    resets_timed = int(rs.item())

    if rank == 0:
        alg = algorithmic_bytes_per_env_step(w["n"], w["m"], w["k"], A)
        peaks_file = ROOT / "MEASURED_PEAKS.json"
        if peaks_file.exists():
            peak, peak_src = float(json.loads(peaks_file.read_text())["hbm_gbs"]), "of measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = 6650.0, "of fallback (B200_PROFILING.md 6.65 TB/s)"
        achieved = alg * B / (kernel_ms * 1e-3) / 1e9          # rank 0's own kernel time
        traffic, traffic_src = None, None
        tf = ROOT / "profiles" / "traffic.json"
        if tf.exists():
            try:
                rec = json.loads(tf.read_text()).get(f"{wname}:{B}")      # committed ncu capture for this shape and batch
                if rec:
                    traffic = rec["dram_bytes_per_launch"]
                    traffic_src = (f"ncu --set full capture {rec.get('source', 'profiles/')} of this kernel at this "
                                   f"shape and batch (committed; NOT measured in this run)")
            except Exception:
                traffic = None
        value = Bg * K / (ms * 1e-3)
        d = bank.plan.dims
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "u32", "data": "synthetic",
            "config": {"workload": f"{wname}: uniform random {w['k']}-SAT n={w['n']} m={w['m']}, {A} agents x {V} vars, "
                                   f"obs_dim {env.obs_dim}, {Bg} envs sharded over {world} GPU(s) ({B} on rank 0), "
                                   f"{P} distinct formulas, max_steps {MAX_STEPS}, auto-reset on (episodes de-phased: "
                                   f"env g starts at step g mod {MAX_STEPS}), action_mode 0",
                       "envs_global": Bg, "envs_per_gpu": B, "problems": P,
                       "group_threads": d.group_threads,
                       "launch": {"step": "one kernel launch per step (msat_rollout_step)",
                                  "graph": f"one kernel launch per step, replayed as CUDA graphs of {G} steps",
                                  "multi": f"msat_rollout_steps: {G} steps per launch, observations of every step "
                                           f"written to [K,B,A,D]"}[mode],
                       "l2": f"no flush: each step writes {B * A * env.obs_dim * 4 / 1e6:.0f} MB of observations per GPU "
                             f"(> 126 MB L2) and cycles {ACTION_CYCLE} action batches"
                             if B * A * env.obs_dim * 4 > 126e6 else
                             f"no flush and the per-step working set ({B * A * env.obs_dim * 4 / 1e6:.0f} MB of "
                             f"observations per GPU) fits the 126 MB L2: writes may be absorbed by L2"},
            "autoreset_in_timed_region": {"resets": resets_timed, "env_steps": Bg * K,
                                          "frac": resets_timed / float(Bg * K)},
            "autoreset_frac_in_timed_region": resets_timed / float(Bg * K),
            "clocks": sampler.summary(t_wall0, t_wall1),
            "e2e": {"value": Bg * Ke / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d * world,
                    "d2h_bytes_per_step": d2h * world, "steps": Ke, "wall_ms_per_step": e2e_wall_ms / Ke,
                    "what": "VecSATEnv.step_host_async -> msat_rollout_step_host_async (depth-2 pipeline): every step "
                            "uploads a pinned host action batch, runs the fused step and downloads team reward, "
                            "done, solved, num_unsatisfied, episode_step into pinned host memory; the host reads "
                            "the results of step t-2 while steps t-1 / t are in flight; observations stay in HBM "
                            "for the policy"},
            "e2e_sync": {"value": Bg * Ks / (e2e_sync_ms * 1e-3), "unit": UNIT, "steps": Ks,
                         "what": "msat_rollout_step_host: one blocking call per step (upload, step, download, stream "
                                 "synchronise), results expanded to the reference's per-agent dicts as views"},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "kernel": "msat::env_kernel<GS, MODE_STEP, OBS> (msat_rollout_step)",
                         "kernel_ms": kernel_ms, "algorithmic_bytes_per_env_step": alg, "envs_per_launch": B,
                         "achieved_dram_gbs": None if traffic is None else traffic / (kernel_ms * 1e-3) / 1e9,
                         "note": "achieved = SURVEY 8(d) algorithmic bytes (int32 literals counted at 4 B each) / "
                                 "kernel time; the kernel reads the formula as packed u16 codes, so its real DRAM "
                                 "traffic is ~3 % below the algorithmic figure and frac can read slightly above 1 "
                                 "when the kernel sits at the copy bandwidth"},
        }
        if reset_legs:
            reset_legs["reset_heavy"]["ms_per_step"] = heavy_ms
            reset_legs["all_reset"]["ms_per_step"] = allr_ms
            for v in reset_legs.values():
                v["value"] = Bg / (v["ms_per_step"] * 1e-3)
            line["reset_heavy"] = reset_legs["reset_heavy"]
            line["all_reset"] = reset_legs["all_reset"]
        if e2e_obs:
            line["e2e_obs_to_host"] = {"value": Bg * args.e2e_obs_steps / (e2e_obs_ms * 1e-3), "unit": UNIT,
                                       "d2h_bytes_per_step": (d2h + e2e_obs[1]) * world, "steps": args.e2e_obs_steps,
                                       "what": "as e2e_sync, plus the int32 observations copied to pinned host memory"}
        if kstep_info:
            line["multi_step_launch"] = kstep_info
        if gnn_info:
            gnn_info["frac_of_hbm_peak"] = gnn_info["gbs"] / peak
            line["gnn_input_mode"] = gnn_info
        if i8_info:
            i8_info["frac_of_hbm_peak"] = i8_info["gbs"] / peak
            line["obs_int8_mode"] = i8_info
        if gae_info:
            gae_info["scan_ms"], gae_info["normalize_ms"] = scan_ms_max, norm_ms_max
            gae_info["scan_gbs"] = 17.0 * gae_info["num_steps"] * B / (scan_ms_max * 1e-3) / 1e9
            gae_info["normalize_gbs"] = 8.0 * gae_info["num_steps"] * B / (norm_ms_max * 1e-3) / 1e9
            gae_info["scan_frac_of_hbm_peak"] = gae_info["scan_gbs"] / peak
            gae_info["normalize_frac_of_hbm_peak"] = gae_info["normalize_gbs"] / peak
            line["gae"] = gae_info
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"], _ = run_cpu_restatement(wname, args.cpu_envs_per_core, 5, 1)
            try:        # BASELINE configs[0]: the reference's own CPU-runnable case (uf20-91 x 16 envs)
                c1, _ = run_cpu_restatement_c("uf20-91", 1, 200, 10, total_envs=16)
                line["cpu_baseline_c1"] = c1
            except Exception as e:
                line["cpu_baseline_c1"] = {"error": repr(e)}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    vec_h.close()
    return 0


def parse_args(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", choices=sorted(WORKLOADS), default="uf100-430")
    ap.add_argument("--envs", type=int, default=0, help="global env count (default: the workload's)")
    ap.add_argument("--problems", type=int, default=0, help="distinct formulas in the bank (default: = envs)")
    ap.add_argument("--scaling", choices=["strong", "weak"], default="strong",
                    help="strong: the global batch is fixed and sharded (BASELINE configs[2]); weak: per-GPU batch fixed")
    ap.add_argument("--group-threads", type=int, default=0)
    ap.add_argument("--e2e-steps", type=int, default=50)
    ap.add_argument("--e2e-obs-steps", type=int, default=2)
    ap.add_argument("--cpu-envs-per-core", type=int, default=128)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gae", action="store_true")
    ap.add_argument("--no-gnn-leg", action="store_true")
    ap.add_argument("--launch", choices=["auto", "step", "graph", "multi"], default="auto",
                    help="how the timed rollout steps are launched: one launch per step, CUDA graphs of 32 steps, or "
                         "32 fused steps per launch (msat_rollout_steps); auto picks by per-GPU batch size")
    ap.add_argument("--graph", type=int, default=-1, metavar="G",
                    help="G > 0: CUDA graphs of G steps each; 0: never use graphs; default -1: follow --launch")
    ap.add_argument("--no-reset-legs", action="store_true")
    ap.add_argument("--no-kstep-leg", action="store_true")
    ap.add_argument("--gae-steps", type=int, default=512, help="T of the GAE leg (configs/MAPPO_CONFIG.yaml NUM_STEPS)")
    ap.add_argument("--emulate-shard", type=int, nargs=2, metavar=("WORLD", "RANK"), default=None,
                    help="debug: single process, but own the env shard of RANK out of WORLD")
    ap.add_argument("--watchdog", type=int, default=420,
                    help="seconds after which all thread stacks are dumped to stderr and the process exits")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last one (obs, reward, done, solved, "
                         "num_unsatisfied, episode_step; rank 0's envs) as DIR/<name>.npy in float32; above 64 MB "
                         "a fixed, seeded sample of env rows, listed in DIR/env_index.npy")
    args = ap.parse_args(argv)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


def _guard_stdout():
    """Keep the real stdout for the ONE JSON line and point fd 1 at stderr so that library chatter
    (e.g. NCCL's version banner) cannot land in front of it."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


if __name__ == "__main__":
    a = parse_args()
    if a.watchdog > 0:      # never hang the caller: dump every thread's stack and exit
        import faulthandler
        faulthandler.dump_traceback_later(a.watchdog, exit=True)
    _json_out = _guard_stdout()
    _print = print

    def print(*args, **kw):  # noqa: A001  (the JSON line goes to the real stdout)
        kw.setdefault("file", _json_out)
        _print(*args, **kw)
        kw["file"].flush()

    sys.exit(main_reference(a) if a.impl == "reference" else main_ours(a))
