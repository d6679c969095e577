"""ctypes binding of libmarlsat_b200.so (the C ABI declared in include/marl_sat_b200.h).

There is no CPU fallback: importing this module without the built library raises, and every
enqueue call needs a CUDA device.  Build with ``python marl_sat_b200/build.py`` (or
``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

from .build import LIB_PATH

MSAT_OK, MSAT_EINVAL, MSAT_EALIGN, MSAT_EUNSUPPORTED = 0, -1, -2, -3
_ERR = {MSAT_EINVAL: "MSAT_EINVAL (bad shape / null pointer / out-of-range scalar)",
        MSAT_EALIGN: "MSAT_EALIGN (buffer not aligned as documented)",
        MSAT_EUNSUPPORTED: "MSAT_EUNSUPPORTED (shape exceeds one CTA's shared memory)"}


class MsatError(RuntimeError):
    pass


class Dims(C.Structure):
    _fields_ = [(name, C.c_int32) for name in
                ("n", "m", "k", "A", "V", "D", "action_mode", "max_steps", "rec_bytes", "state_words",
                 "group_threads", "smem_bytes")]


_p = C.c_void_p
_i32 = C.c_int32
_i64 = C.c_int64
_f64 = C.c_double

# name -> (restype, argtypes); mirrors include/marl_sat_b200.h one to one
SIGNATURES = {
    "msat_version": (C.c_char_p, []),
    "msat_num_agents_for": (_i32, [_i32, _i32]),
    "msat_plan_create": (C.c_int, [C.POINTER(_p), _i32, _i32, _i32, _i32, _i32, _i32, _i32]),
    "msat_plan_destroy": (None, [_p]),
    "msat_plan_dims": (C.c_int, [_p, C.POINTER(Dims)]),
    "msat_compile_bank": (C.c_int, [_p, _p, _i32, _p, _p]),
    "msat_reset": (C.c_int, [_p, _p, _i32, _p, _p, _p, _p, _i32, _p]),
    "msat_import_state": (C.c_int, [_p, _p, _i32, _p, _p, _p, _p, _p, _p, _i32, _p]),
    "msat_plan_set_reward": (C.c_int, [_p, _i32, _f64, _f64, _f64]),
    "msat_tune": (C.c_int, [C.c_char_p, _i32]),
    "msat_plan_set_reset_counter": (C.c_int, [_p, _p]),
    "msat_plan_set_clause_update": (C.c_int, [_p, _i32]),
    "msat_plan_set_obs_dtype": (C.c_int, [_p, _i32]),
    "msat_step": (C.c_int, [_p, _p, _i32, _p, _p, _p, _i32, _p, _p, _p, _p, _i32, _p, _i32, _p, _p, _p, _p, _i32, _p]),
    "msat_rollout_steps": (C.c_int, [_p, _p, _i32, _p, _p, _p, _i32, _p, _p, _i32, _i32, _p, _p, _p, _i32, _p, _i32,
                                     _p, _i32, _p, _p, _p, _p, _i32, _p]),
    "msat_host_pipe_create": (C.c_int, [C.POINTER(_p), _i32]),
    "msat_host_pipe_destroy": (None, [_p]),
    "msat_rollout_step_host_async": (C.c_int, [_p, _i32, _p, _p, _i32, _p, _p, _p, _p, _p, _i32, _i32, _p, _p, _i32, _p,
                                               _i32, _p, _p, _p] + [_p] * 5 + [_i32, _p]),
    "msat_host_wait": (C.c_int, [_p, _i32]),
    "msat_shutdown": (C.c_int, []),
    "msat_rollout_step": (C.c_int, [_p, _p, _i32, _p, _p, _p, _p, _p, _i32, _i32, _p, _p, _i32, _p, _i32, _p, _p, _p, _i32, _p]),
    "msat_rollout_step_gnn": (C.c_int, [_p, _p, _i32, _p, _p, _p, _p, _p, _i32, _i32, _p, _p, _p, _i32, _p, _i32, _p, _p, _p, _i32, _p]),
    "msat_get_obs": (C.c_int, [_p, _p, _i32, _p, _p, _i32, _p]),
    "msat_export_state": (C.c_int, [_p, _p, _i32, _p, _i32] + [_p] * 10 + [_p]),
    "msat_rollout_step_host": (C.c_int, [_p, _p, _i32, _p, _p, _p, _p, _p, _i32, _i32, _p, _p, _i32, _p, _i32, _p, _p, _p] + [_p] * 5 + [_i32, _p]),
    "msat_rng_chain": (C.c_int, [_p, _p, _p]),
    "msat_rng_split2": (C.c_int, [_p, _p, _p]),
    "msat_env_keys": (C.c_int, [_p, _p, _i32, _i32, _i32, _i32, _p, _p, _p]),
    "msat_env_keys_weighted": (C.c_int, [_p, _p, _i32, _i32, _i32, _p, _i32, _p, _p, _p]),
    "msat_problem_stats": (C.c_int, [_p, _i64, _i64, _p, _p, _p, _p, _i32, _i32, _i32, _p, _p]),
    "msat_gae": (C.c_int, [_p, _i64, _i64, _p, _p, _p, _f64, _f64, _p, _p, _p, _i32, _i32, _p]),
    "msat_adv_stats": (C.c_int, [_p, _i64, _p, _p]),
    "msat_adv_normalize": (C.c_int, [_p, _i64, _p, _p]),
    "msat_gnn_static": (C.c_int, [_p, _p, _i32, _p, _p, _p, _p]),
    "msat_gnn_dynamic": (C.c_int, [_p, _p, _i32, _p, _i32, _p, _p, _p]),
    "msat_rollout_metrics": (C.c_int, [_p, _i64, _i64, _p, _p, _p, _p, _i32, _i32, _p, _p]),
    "msat_flip_gains": (C.c_int, [_p, _p, _i32, _p, _i32, _f64, _p, _p, _p]),
    "msat_dimacs_parse": (C.c_int, [C.c_char_p, C.c_size_t, _i32, C.POINTER(_i32), C.POINTER(_i32), C.POINTER(_i32),
                                    C.POINTER(_i32), _p, _i32]),
    "msat_eval_track": (C.c_int, [_p, _p, _p, _i32, _i32, _p, _p, _p, _p]),
    "msat_walksat": (C.c_int, [_p, _p, _i32, _p, _p, _i32, _i32, _f64, _p, _p, _i32, _p]),
    "msat_obs_compression": (C.c_int, [C.c_int, C.POINTER(C.c_int)]),
    "msat_obs_alloc": (_p, [C.c_size_t, C.c_int, _p]),
    "msat_obs_free": (None, [_p, C.c_size_t, C.c_int, _p]),
}

_lib = None


def lib_path() -> Path:
    return LIB_PATH


def load() -> C.CDLL:
    """Load the shared library (once).  Fails loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is missing: the CUDA library has not been built and marl_sat_b200 has no CPU "
            f"fallback. Run `python marl_sat_b200/build.py` (needs nvcc).")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        if not hasattr(lib, name):
            continue          # optional next-tier entry points are bound only when present
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc == MSAT_OK:
        return
    if rc < 0:
        raise MsatError(f"{what}: {_ERR.get(rc, rc)}")
    raise MsatError(f"{what}: CUDA error {rc} (cudaError_t)")
