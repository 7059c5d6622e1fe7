"""Builds libgnc.so (the C-ABI CUDA library, include/gnc.h) in-tree with nvcc for sm_100a.

Called by ``__graft_entry__.build()`` and usable stand-alone:
    python -m graphnet_classifier_b200.build [--force]
nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU
box with the repo snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libgnc.so")
SOURCES = ["graph_build.cu", "aggregate.cu", "dense.cu", "tc_linear.cu", "tc_chain.cu", "tc_wgrad.cu", "tc_bwd.cu", "train_ops.cu", "narrow.cu", "slic.cu", "slic_connect.cu", "resize.cu", "jpeg.cu", "png.cu"]
NVCC_FLAGS = [
    "-O3", "-std=c++17",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "--threads", "0",
    "-Xcompiler", "-fPIC", "-shared", "-Xcompiler", "-pthread",
    "-Xcompiler", "-ffp-contract=off",      # host: the resize coefficient tables follow Pillow's double arithmetic
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC or put /usr/local/cuda/bin on PATH)")


def _stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    deps.append(os.path.join(os.path.dirname(PKG_DIR), "include", "gnc.h"))
    return any(os.path.getmtime(d) > t for d in deps if os.path.isfile(d))


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB_PATH
    cmd = [_nvcc(), *NVCC_FLAGS, "-o", LIB_PATH] + [os.path.join(CSRC, s) for s in SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    res = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
