"""Time msat_import_state against msat_reset at the headline shape (uf100-430 x 65,536 envs, one formula per env).

Both build a fresh packed state on the same formulas and write the same outputs; the import reads the assignment
(int32[n]), step and done flag of every env from memory where the reset draws the assignment with Threefry.  Three
cases: int32 observations, int8 observations, no observations.  Per case the two launches alternate in blocks of
`--per-block` back-to-back launches between CUDA events on one stream, after a warm-up; the reported time per launch is
the median over the blocks.  The output (4.1 GB of int32 observations per launch) is far larger than the 126 MB L2.

Algorithmic bytes per env (what each launch has to move at least):
  reset   problem index 4 + key 8 + formula record (literals + agent-mask stream with observations, literals only
          without) + state record + observations
  import  problem index 4 + assignment 4n + step 4 + done 1 + the same record, state and observations
Fraction of peak = bytes / time over the measured 6,546.6 GB/s device copy bandwidth (DESIGN.md section 4).

    python profiles/import_state_bench.py [--envs 65536] [--blocks 30] [--per-block 5] [--out result.json]
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

PEAK_GBS = 6546.6


def power_limit() -> str:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return out.stdout.strip() or "unknown"
    except Exception:
        return "unknown"


def run_case(M, obs_dtype, want_obs, B, n, m, blocks, per_block, seed=0):
    from marl_sat_b200.env import _ptr
    from marl_sat_b200.synth import uniform_ksat
    dev = torch.device("cuda")
    env = M.SATEnv(n, m, 512, verbose=False, obs_dtype=obs_dtype)
    bank = env.make_bank(torch.from_numpy(uniform_ksat(B, n, m, 3, seed)))
    d = bank.plan.dims
    g = torch.Generator(device=dev).manual_seed(seed)
    idx = torch.randperm(B, generator=g, device=dev).to(torch.int32)
    keys = torch.randint(-2 ** 31, 2 ** 31 - 1, (B, 2), generator=g, device=dev, dtype=torch.int64).to(torch.int32)
    assign = torch.randint(0, 2, (B, n), generator=g, device=dev, dtype=torch.int32)
    step = torch.randint(0, 512, (B,), generator=g, device=dev, dtype=torch.int32)
    done = torch.zeros(B, dtype=torch.uint8, device=dev)
    state = torch.empty((B, d.state_words), dtype=torch.int32, device=dev)
    obs = torch.empty((B, d.A, d.D), dtype=env.obs_dtype, device=dev) if want_obs else None
    lib, plan, stream = env._lib, bank.plan.handle, torch.cuda.current_stream(dev).cuda_stream
    reset_args = (plan, _ptr(bank.data), B, _ptr(idx), _ptr(keys), _ptr(state), _ptr(obs), B, stream)
    import_args = (plan, _ptr(bank.data), B, _ptr(idx), _ptr(assign), _ptr(step), _ptr(done), _ptr(state), _ptr(obs),
                   B, stream)
    launch = {"reset": lambda: lib.msat_reset(*reset_args), "import": lambda: lib.msat_import_state(*import_args)}

    # the import of the reset's own assignment reproduces the reset's packed state (and observations)
    assert launch["reset"]() == 0
    ref_state, ref_obs = state.clone(), (obs.clone() if want_obs else None)
    exported = M.SATState(env, bank, ref_state, True).variable_assignments
    env.import_state(bank, idx, exported, state_out=state, obs_out=obs, want_obs=want_obs)
    assert torch.equal(state, ref_state) and (not want_obs or torch.equal(obs, ref_obs))
    del ref_obs, exported

    for _ in range(3):
        for name in ("reset", "import"):
            for _ in range(per_block):
                assert launch[name]() == 0
    torch.cuda.synchronize()
    times = {"reset": [], "import": []}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4 * blocks)]
    for b in range(blocks):
        order = ("reset", "import") if b % 2 == 0 else ("import", "reset")
        for j, name in enumerate(order):
            e0, e1 = ev[4 * b + 2 * j], ev[4 * b + 2 * j + 1]
            e0.record()
            for _ in range(per_block):
                launch[name]()
            e1.record()
            times[name].append((e0, e1))
    torch.cuda.synchronize()
    rec = d.rec_bytes  # stride; the launch stages only the leading part of a record
    lits_bytes = (((m + 1) & ~1) * d.k * 2 + 15) & ~15
    fw1 = (d.A * d.D + 31) // 32 + 1
    rec_read = ((lits_bytes + 4 * fw1 + 15) & ~15) if want_obs else lits_bytes
    obs_bytes = d.A * d.D * (1 if obs_dtype == "int8" else 4) if want_obs else 0
    common = rec_read + 4 * d.state_words + obs_bytes + 4
    bytes_env = {"reset": common + 8, "import": common + 4 * n + 4 + 1}
    res = {}
    for name in ("reset", "import"):
        per_launch = [e0.elapsed_time(e1) / per_block for e0, e1 in times[name]]
        ms = statistics.median(per_launch)
        gbs = bytes_env[name] * B / (ms * 1e-3) / 1e9
        res[name] = {"ms_per_launch_median": round(ms, 5), "ms_min": round(min(per_launch), 5),
                     "ms_max": round(max(per_launch), 5), "bytes_per_env": bytes_env[name],
                     "achieved_gbs": round(gbs, 1), "frac_of_measured_peak": round(gbs / PEAK_GBS, 4)}
    res["import_over_reset"] = round(res["import"]["ms_per_launch_median"] / res["reset"]["ms_per_launch_median"], 4)
    res["group_threads"] = d.group_threads if want_obs else "launch without observations (one warp per env)"
    res["record_stride_bytes"] = rec
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--blocks", type=int, default=30, help="timed blocks per launch kind (alternating)")
    ap.add_argument("--per-block", type=int, default=5, help="back-to-back launches per timed block")
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: this measurement has no CPU fallback")
    import marl_sat_b200 as M
    n, m, B = 100, 430, args.envs
    result = {"what": "msat_import_state vs msat_reset, uf100-430", "envs": B, "formulas": B,
              "device": torch.cuda.get_device_name(), "power_limit": power_limit(),
              "timing": f"CUDA events, median over {args.blocks} alternating blocks of {args.per_block} launches, "
                        f"after warm-up", "peak_gbs_measured_copy": PEAK_GBS, "cases": {}}
    for case, (dtype, want_obs) in {"obs_int32": ("int32", True), "obs_int8": ("int8", True),
                                    "no_obs": ("int32", False)}.items():
        result["cases"][case] = run_case(M, dtype, want_obs, B, n, m, args.blocks, args.per_block)
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
            f.write("\n")


if __name__ == "__main__":
    main()
