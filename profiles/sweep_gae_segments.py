import sys
from pathlib import Path
import torch
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import marl_sat_b200 as M
from marl_sat_b200 import _lib
lib = _lib.load()
dev = torch.device("cuda", 0)
T = 512
for B in (2048, 4096, 8192, 16384, 20480):
    g = torch.Generator(device=dev).manual_seed(0)
    reward = (torch.rand((T, B), generator=g, device=dev) < 0.01).float()
    done = (torch.rand((T, B), generator=g, device=dev) < 0.005).to(torch.uint8)
    value = torch.randn((T, B), generator=g, device=dev)
    last = torch.randn((B,), generator=g, device=dev)
    adv, tgt = torch.empty((T, B), device=dev), torch.empty((T, B), device=dev)
    stats = torch.zeros(3, dtype=torch.float64, device=dev)
    for wps in (8, 16, 24, 32, 48, 64):
        lib.msat_tune(b"gae_warps_per_sm", wps)
        for _ in range(3):
            M.calculate_gae(reward, done, value, last, 0.995, 0.95, stats=stats, out=(adv, tgt))
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            for _ in range(10):
                M.calculate_gae(reward, done, value, last, 0.995, 0.95, stats=stats, out=(adv, tgt))
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); gr.replay(); e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1) / 10)
        print(f"B={B:6d} warps/SM target {wps:3d}: {best*1e3:7.1f} us  frac {17.0*T*B/(best*1e-3)/1e9/6546.6:.3f}")
