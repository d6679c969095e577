"""Observation buffers in compressible device memory (``obs_empty`` / ``msat_obs_alloc``): every entry point writes
the same bits there as into ordinary memory, graph capture works, the free path returns the memory, and a B200
grants the compression."""
import ctypes as C

import pytest
import torch

from oracle import threefry as otf

pytestmark = pytest.mark.gpu


def _msat():
    import marl_sat_b200 as M
    return M


def _pool():
    from marl_sat_b200.env import _obs_pool
    return _obs_pool(torch.device("cuda", torch.cuda.current_device()))


def _in_pool(t: torch.Tensor) -> bool:
    pool = _pool()
    if pool is None:
        return False
    snap = pool.snapshot()
    segments = snap["segments"] if isinstance(snap, dict) else snap
    p = t.data_ptr()
    return any(s["address"] <= p < s["address"] + s["total_size"] for s in segments)


def _ordinary(t: torch.Tensor) -> torch.Tensor:
    o = torch.empty(t.shape, dtype=t.dtype, device=t.device)
    assert not _in_pool(o)
    return o


def test_b200_grants_compression():
    from marl_sat_b200 import _lib
    granted = C.c_int(-1)
    assert _lib.load().msat_obs_compression(torch.cuda.current_device(), C.byref(granted)) == 0
    assert _lib.load().msat_obs_compression(-1, C.byref(granted)) == _lib.MSAT_EINVAL
    if "B200" not in torch.cuda.get_device_name():
        pytest.skip("compression is required on a B200 only")
    assert granted.value == 1, "a B200 must grant generic compression for observation buffers"
    assert _pool() is not None
    M = _msat()
    env = M.SATEnv(20, 91, 8, verbose=False)
    assert _in_pool(env.alloc_step_outputs(4)["obs"])


# (n, m, vars per agent, envs, obs dtype, K of the multi-step launch)
SHAPES = [
    (100, 430, None, 65536, "int32", 2),      # the headline shape
    (100, 430, None, 65536, "int8", 2),
    (20, 91, None, 77, "int32", 5),           # half-warp groups; D = 131 rows are not 16-byte multiples
    (20, 91, None, 77, "int8", 5),
    (35, 149, 7, 41, "int32", 3),
]


@pytest.mark.parametrize("n,m,vpa,B,dtype,K", SHAPES)
def test_compressible_obs_are_bit_identical(n, m, vpa, B, dtype, K):
    M = _msat()
    from marl_sat_b200.synth import uniform_ksat_torch
    dev = torch.device("cuda", torch.cuda.current_device())
    env = M.SATEnv(n, m, 6, vars_per_agent=vpa, verbose=False, obs_dtype=dtype)
    bank = env.make_bank(uniform_ksat_torch(min(B, 4096), n, m, 3, seed=n + B, device=dev))
    key = otf.prng_key(7)
    comp, plain = M.VecSATEnv(env, bank, B, key), M.VecSATEnv(env, bank, B, key)
    plain.out["obs"] = _ordinary(plain.out["obs"])
    if _pool() is not None:
        assert _in_pool(comp.out["obs"])
    # reset
    assert torch.equal(comp.reset(), plain.reset())
    # single steps, auto-reset included (max_steps 6)
    g = torch.Generator(device=dev).manual_seed(B)
    acts = torch.randint(0, env.max_vars_per_agent + 1, (8, B, env.num_agents), generator=g, device=dev,
                         dtype=torch.int32)
    for t in range(8):
        a, b = comp.step(acts[t]), plain.step(acts[t])
        assert torch.equal(a["obs"], b["obs"]), f"step {t}"
        assert torch.equal(a["reward"], b["reward"]) and torch.equal(a["done"], b["done"])
    # msat_rollout_steps with every step's observations
    oc, op = comp.alloc_multi_step_outputs(K, emit_every_step=True), plain.alloc_multi_step_outputs(K, emit_every_step=True)
    op["obs"] = _ordinary(op["obs"])
    comp.steps(acts[:K], oc)
    plain.steps(acts[:K], op)
    assert torch.equal(oc["obs"], op["obs"]) and torch.equal(oc["reward"], op["reward"])
    # get_obs into a compressible buffer against msat_get_obs into an ordinary one
    got = env.get_obs_array(comp.sat_state())
    ref = _ordinary(got)
    assert env._lib.msat_get_obs(bank.plan.handle, bank.data.data_ptr(), bank.num_problems, plain.state.data_ptr(),
                                 ref.data_ptr(), B, torch.cuda.current_stream().cuda_stream) == 0
    assert torch.equal(got, ref) and torch.equal(got, op["obs"][K - 1])
    assert torch.equal(comp.state, plain.state)


def test_graph_replay_into_compressible_obs():
    M = _msat()
    from marl_sat_b200.synth import uniform_ksat_torch
    dev = torch.device("cuda", torch.cuda.current_device())
    env = M.SATEnv(50, 218, 5, verbose=False)
    bank = env.make_bank(uniform_ksat_torch(64, 50, 218, 3, seed=3, device=dev))
    B, G = 1000, 6
    graphed, eager = M.VecSATEnv(env, bank, B, otf.prng_key(1)), M.VecSATEnv(env, bank, B, otf.prng_key(1))
    eager.out["obs"] = _ordinary(eager.out["obs"])
    graphed.reset()
    eager.reset()
    acts = torch.randint(0, env.max_vars_per_agent + 1, (G, B, env.num_agents), device=dev, dtype=torch.int32)
    state0, chain0, cur0 = graphed.state.clone(), graphed.keys._bufs.clone(), graphed.keys._cur
    for t in range(G):                     # warm-up outside the capture, then put the env back
        graphed.step(acts[t])
    graphed.state.copy_(state0)
    graphed.keys._bufs.copy_(chain0)
    graphed.keys._cur = cur0
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for t in range(G):
            graphed.step(acts[t])
    graphed.state.copy_(state0)
    graphed.keys._bufs.copy_(chain0)
    graph.replay()
    for t in range(G):
        eager.step(acts[t])
    torch.cuda.synchronize()
    assert torch.equal(graphed.out["obs"], eager.out["obs"])
    assert torch.equal(graphed.state, eager.state)


def test_free_path_returns_the_memory():
    if _pool() is None:
        pytest.skip("the device does not grant compressible memory")
    from marl_sat_b200 import _lib
    from marl_sat_b200.env import obs_empty
    dev = torch.device("cuda", torch.cuda.current_device())
    n = 1 << 30                                                 # 4 GiB of int32
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free0 = torch.cuda.mem_get_info(dev)[0]
    for i in range(20):
        t = obs_empty((n,), torch.int32, dev)
        t.fill_(i - 1)
        assert int(t[n - 1]) == i - 1
        del t
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    # the pool lives as long as the process and may keep one freed buffer cached, but never one per allocation
    free1 = torch.cuda.mem_get_info(dev)[0]
    assert free1 >= free0 - 4 * n - (64 << 20), (free0, free1)
    # a pool of the same allocator that goes away hands its memory back through msat_obs_free
    alloc = torch.cuda.memory.CUDAPluggableAllocator(str(_lib.lib_path()), "msat_obs_alloc", "msat_obs_free")
    for _ in range(20):
        pool = torch.cuda.MemPool(alloc.allocator())
        with torch.cuda.use_mem_pool(pool, dev):
            t = torch.empty((n,), dtype=torch.int32, device=dev)
        t.zero_()
        del t
        torch.cuda.synchronize()
        del pool
    torch.cuda.empty_cache()
    free2 = torch.cuda.mem_get_info(dev)[0]
    assert free2 >= free1 - (64 << 20), (free1, free2)
