"""Build libraymond_cuda.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m raymond_b200.build [--force] [--verbose]
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libraymond_cuda.so")
SOURCES = ["rm_host.cpp", "rm_project.cpp", "rm_task.cpp", "rm_device.cu", "rm_gridbuild.cu", "rm_display.cu"]
HEADERS = ["rm_internal.hpp", "rm_kernels.cuh", os.path.join("..", "..", "include", "raymond.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    # rustc never contracts a*b+c; the reference's f64 decision sequence is replayed one IEEE op at a time
    "-fmad=false",
    "-Xcompiler", "-fPIC,-O2,-ffp-contract=off,-Wall,-pthread",
    "-shared", "-cudart", "shared",
]


def nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; raymond_b200 has no CPU build")


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def build(force: bool = False, verbose: bool = False, defines=(), out: str = LIB) -> str:
    """`defines` / `out` build an instrumented library next to the default one: defines=["RM_TRAV_PROFILE"],
    out=".../trav_profile.so" adds k_traverse's per-phase cycle counters (read by scripts/trav_profile.py)."""
    if not force and out == LIB and not needs_build():
        return LIB
    cmd = [nvcc()] + NVCC_FLAGS + [f"-D{d}" for d in defines] + (["-Xptxas", "-v"] if verbose else []) + \
          [os.path.join(CSRC, f) for f in SOURCES] + ["-o", out]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed building libraymond_cuda.so")
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
