"""Builds the C-ABI shared library (`x3d_tf_b200/lib/libx3d_b200.so`) with nvcc for sm_100a.

In-tree build so that the `.so` travels with the repository snapshot to the GPU box; nvcc
cross-compiles without a GPU.  `python -m x3d_tf_b200.build [--force]`.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libx3d_b200.so")
SOURCES = ["host_util.cu", "x3d_simt.cu", "x3d_pw_tc.cu", "x3d_pw_tf32_tc.cu", "x3d_dw_tma.cu", "x3d_dw_planar.cu", "x3d_stem_tc.cu", "x3d_ab_fused.cu", "x3d_ab_persist.cu", "x3d_train.cu", "x3d_io.cu", "x3d_jpeg.cu", "x3d_jpeg_enc.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=default",
              "--expt-relaxed-constexpr"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(LIB_DIR, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(HERE, "..", "include", "x3d_b200.h"))
    objs, jobs = [], []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(LIB_DIR, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + headers):
            cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
            if verbose:
                print(" ".join(cmd))
            jobs.append(subprocess.Popen(cmd))
    failed = [j.args for j in jobs if j.wait() != 0]
    if failed:
        raise subprocess.CalledProcessError(1, failed[0])
    if force or _stale(LIB_PATH, objs):
        cmd = [_nvcc(), "-shared", "-o", LIB_PATH] + objs + ["-cudart", "static"]
        if verbose:
            print(" ".join(cmd))
        subprocess.run(cmd, check=True)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv or "--verbose" in sys.argv))
