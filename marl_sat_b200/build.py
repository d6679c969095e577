"""In-tree build of libmarlsat_b200.so (hand-written CUDA for sm_100a, C ABI in include/marl_sat_b200.h).

The library is compiled with plain ``nvcc`` (no torch extension machinery): the boundary is a C ABI and
the Python layer binds it with ctypes.  ``python marl_sat_b200/build.py`` rebuilds it (run as a script so the package, which refuses to import
without the library, is not imported first).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

CSRC = Path(__file__).resolve().parent / "csrc"
LIB_PATH = CSRC / "libmarlsat_b200.so"
SOURCES = ["cabi.cu", "satenv.cu", "keys.cu", "gae.cu", "features.cu", "local_search.cu", "obs_memory.cu", "sampling.cu",
           "dimacs.cpp"]
HEADERS = ["common.cuh", "internal.h", "../../include/marl_sat_b200.h"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found: cannot build libmarlsat_b200.so (set NVCC=/path/to/nvcc)")


def is_stale() -> bool:
    if not LIB_PATH.exists():
        return True
    t = LIB_PATH.stat().st_mtime
    deps = [CSRC / s for s in SOURCES if (CSRC / s).exists()] + [(CSRC / h).resolve() for h in HEADERS]
    return any(p.stat().st_mtime > t for p in deps if p.exists())


def build(force: bool = False, verbose: bool = False) -> Path:
    """Compile every ``.cu`` under ``csrc/`` into one shared library for sm_100a."""
    if not force and not is_stale():
        return LIB_PATH
    srcs = [s for s in SOURCES if (CSRC / s).exists()]
    cmd = [_nvcc(), *NVCC_FLAGS] + (["-Xptxas", "-v"] if verbose else []) + ["-o", str(LIB_PATH), *srcs]
    res = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stdout + res.stderr)
    return LIB_PATH


FFI_SRC = CSRC / "xla_ffi_shim.cc"
FFI_LIB = CSRC / "libmarlsat_b200_xla.so"


def build_ffi_shim() -> Path:
    """Compile the XLA FFI custom-call layer (csrc/xla_ffi_shim.cc) against the headers JAX ships
    (``jax.ffi.include_dir()``) and link it to libmarlsat_b200.so.  Only possible where JAX >= 0.4.38 is
    installed -- it is not in this image, where the shim is syntax-checked against tests/ffi_stub instead."""
    try:
        from jax import ffi as jffi
    except Exception as e:
        raise RuntimeError("the XLA FFI shim needs JAX (jax.ffi.include_dir()); skipping") from e
    build()
    cmd = [_nvcc(), "-O2", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "-I", jffi.include_dir(), "-o", str(FFI_LIB),
           str(FFI_SRC), "-L", str(CSRC), "-lmarlsat_b200", "-Xlinker", "-rpath", "-Xlinker", "$ORIGIN"]
    res = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("building the XLA FFI shim failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    return FFI_LIB


if __name__ == "__main__":
    print(build(force=True, verbose="-v" in sys.argv))
    if "--ffi" in sys.argv:
        print(build_ffi_shim())
