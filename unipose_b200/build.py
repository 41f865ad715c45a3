"""Builds libunipose_b200.so (hand-written sm_100a CUDA + the C-ABI) in-tree with nvcc.

The shared object is git-ignored but travels with the working tree (so a GPU box without
/root/.cache still finds it).  `python -m unipose_b200.build` forces a rebuild.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_DIR = os.path.join(_HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libunipose_b200.so")
SOURCES = ["conv_tcgen05.cu", "conv_wgrad_tcgen05.cu", "wasp_chain.cu", "bneck_chain.cu", "bneck_tail.cu", "elementwise.cu", "video_eval.cu", "train.cu", "pack_multi.cu", "data_pipeline.cu", "image_prep.cu", "c_api.cu"]
HEADERS = ["up_ptx.cuh", "up_internal.h", "up_conv_host.h", os.path.join("..", "..", "include", "unipose_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (looked at $NVCC, /usr/local/cuda/bin/nvcc, PATH)")


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    lib_m = os.path.getmtime(LIB_PATH)
    for f in SOURCES + HEADERS:
        p = os.path.join(CSRC, f)
        if os.path.exists(p) and os.path.getmtime(p) > lib_m:
            return True
    return False


def build_library(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu of csrc/ into one shared object; returns its path."""
    if not force and not needs_build():
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    tmp = LIB_PATH + ".tmp.%d" % os.getpid()
    cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + srcs + ["-o", tmp]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n%s\n%s" % (" ".join(cmd), res.stdout + res.stderr))
    if verbose:
        sys.stderr.write(res.stdout + res.stderr)
    os.replace(tmp, LIB_PATH)
    return LIB_PATH


if __name__ == "__main__":
    print(build_library(force=True, verbose="-v" in sys.argv))
