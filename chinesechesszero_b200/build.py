"""Build the sm_100a CUDA library in-tree: chinesechesszero_b200/csrc/libccz_b200.so.

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box with the
repo snapshot; there is no JIT cache and no fallback when it is missing.
"""
from __future__ import annotations

import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
OUT = os.path.join(CSRC, "libccz_b200.so")
SOURCES = ["ccz_b200.cu"]
HEADERS = ["ccz_rules.cuh", "ccz_movegen.cuh", "ccz_mcts.cuh", "ccz_replay.cuh", "ccz_conv.cuh", "ccz_stem.cuh", "ccz_heads.cuh", "ccz_dedup.cuh", "../../include/ccz_b200.h"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-shared", "-Xcompiler", "-fPIC",
]


def _nvcc() -> str:
    cand = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    return cand if os.path.exists(cand) else "nvcc"


def is_stale() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def build(force: bool = False, verbose: bool = False) -> str:
    if force or is_stale():
        tmp = OUT + f".tmp{os.getpid()}"
        cmd = [_nvcc(), *NVCC_FLAGS, "-o", tmp, *SOURCES]
        if verbose:
            cmd.insert(1, "-Xptxas")
            cmd.insert(2, "-v")
        subprocess.run(cmd, check=True, cwd=CSRC)
        os.replace(tmp, OUT)
    return OUT


if __name__ == "__main__":
    print(build(force=True, verbose=True))
