"""Builds libcmf_sm100.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo)."""
from __future__ import annotations

import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SO = os.path.join(HERE, "libcmf_sm100.so")
SOURCES = [os.path.join(HERE, "csrc", "cmf_sm100.cu")]
DEPS = SOURCES + [
    os.path.join(HERE, "csrc", "kernels_simt.cuh"),
    os.path.join(HERE, "csrc", "kernels_tc.cuh"),
    os.path.join(HERE, "csrc", "kernels_fd.cuh"),
    os.path.join(HERE, "csrc", "comm.h"),
    os.path.join(HERE, "csrc", "kernels_hals.cuh"),
    os.path.join(HERE, "csrc", "kernels_sparse.cuh"),
    os.path.join(ROOT, "include", "cmf_sm100.h"),
]


def nvcc_path():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def stale():
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in DEPS)


def build(force=False, verbose=False):
    if not force and not stale():
        return SO
    cmd = [
        nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
        "-Xcompiler", "-fPIC", "-shared", "-o", SO, *SOURCES, "-lcuda", "-ldl", "-lpthread",
    ]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    subprocess.check_call(cmd, cwd=ROOT)
    return SO


if __name__ == "__main__":
    print(build(force=True, verbose=True))
