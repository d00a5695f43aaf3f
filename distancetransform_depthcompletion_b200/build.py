"""Builds libdtfill.so (the sm_100a kernels + C ABI) in-tree with nvcc.  nvcc cross-compiles without a GPU."""
from __future__ import annotations

import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(_HERE), "include")
LIB_PATH = os.path.join(_HERE, "libdtfill.so")
SOURCES = ["dtfill.cu"]
HEADERS = sorted(f for f in os.listdir(CSRC) if f.endswith(".cuh")) + [os.path.join(INCLUDE, "dtfill.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + [h if os.path.isabs(h) else os.path.join(CSRC, h) for h in HEADERS]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a into libdtfill.so next to this file; returns the path."""
    if not force and not needs_build():
        return LIB_PATH
    extra = os.environ.get("DTFILL_NVCC_EXTRA", "").split()        # instrumented builds: -DDTFILL_TRACE, -DDTFILL_PLANNER_CLOCKS
    cmd = [_nvcc(), *NVCC_FLAGS, *extra, "-I", INCLUDE, "-I", CSRC, "-o", LIB_PATH] + [os.path.join(CSRC, s) for s in SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force=True, verbose="-v" in __import__("sys").argv))
