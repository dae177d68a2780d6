"""Build libstts_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libstts_b200.so")
SRCS = ["engine.cu"]
DEPS = ["engine.cu", "kernels.cuh", "model.hpp", "conv_tc.cuh", "rb_fused.cuh", "pc_fused.cuh", "nb_fused.cuh", "rng.cuh", "g2p.cuh", "g2p_phases.hpp", os.path.join("..", "..", "include", "stts_b200.h")]


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    for d in DEPS + [os.path.join("..", "build.py")]:
        p = os.path.join(CSRC, d)
        if os.path.exists(p) and os.path.getmtime(p) > t:
            return True
    return False


def build_native(force: bool = False, verbose: bool = False, with_tc: bool | None = None) -> str:
    """nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo ... -> summertts_b200/libstts_b200.so"""
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if with_tc is None:
        with_tc = os.path.exists(os.path.join(CSRC, "conv_tc.cuh")) and os.environ.get("STTS_NO_TC", "0") != "1"
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-shared",
           "-Xcompiler", "-fPIC", "-Xcompiler", "-O2", "-o", LIB] + [os.path.join(CSRC, s) for s in SRCS]
    if with_tc:
        cmd += ["-DSTTS_WITH_TC"]
    if os.environ.get("STTS_TRACE_BUILD", "0") == "1":
        cmd += ["-DSTTS_TC_TRACE_BUILD"]
    if verbose:
        cmd += ["-Xptxas", "-v"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed building libstts_b200.so")
    if verbose:
        sys.stderr.write(r.stdout + r.stderr)
    return LIB


if __name__ == "__main__":
    print(build_native(force=True, verbose="-v" in sys.argv))
