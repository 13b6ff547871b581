"""Builds bspatom_b200/libbspatom.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a."""
from __future__ import annotations

import os
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB = os.path.join(_HERE, "libbspatom.so")
LIB_DEBUG = os.path.join(_HERE, "libbspatom_debug.so")   # -DBSP_DEBUG: device-side bounds / pipeline asserts (tests only)
SOURCES = ["bsp_api.cu"]
HEADERS = ["bsp_api_extra.cuh", "bsp_assembly.cuh", "bsp_core.h", "bsp_driver.h", "bsp_gemm.cuh", "bsp_plan.h",
           "bsp_kernels.cuh", os.path.join("..", "..", "include", "bspatom.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def _stale(lib: str) -> bool:
    if not os.path.exists(lib):
        return True
    t = os.path.getmtime(lib)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def build(force: bool = False, verbose: bool = False, debug: bool = False) -> str:
    lib = LIB_DEBUG if debug else LIB
    if not force and not _stale(lib):
        return lib
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-DBSP_DEBUG"] if debug else []) + (["-Xptxas", "-v"] if verbose else []) + ["-o", lib] + SOURCES
    subprocess.check_call(cmd, cwd=CSRC)
    return lib


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, debug="--debug" in sys.argv))
