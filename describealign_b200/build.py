"""Builds libdescribealign_b200.so in-tree with nvcc for sm_100a.

The library is plain CUDA C++ behind a C ABI (include/describealign_b200.h); it does not
link against torch.  `python -m describealign_b200.build` or __graft_entry__.build().
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libdescribealign_b200.so")
SOURCES = ["api.cu", "features.cu", "stage_a.cu", "stage_b.cu", "traceback.cu", "engine.cu", "pcm_reader.cu", "stretch.cu", "host_stage.cpp"]
HEADERS = ["common.cuh", "dp2_scan.cuh", "refine.cuh", "hann_tables.h", os.path.join("..", "..", "include", "describealign_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-fmad=false",                 # numpy never contracts a*b+c; explicit fma() where OpenBLAS does
    "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-ffp-contract=off", "-Xcompiler", "-mfma",   # host: fma() is one instruction, nothing is contracted
    "-shared",
]


def nvcc_path() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError("nvcc not found: describealign_b200 needs the CUDA toolkit to build")


def is_stale() -> bool:
    if not os.path.isfile(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB
    cmd = [nvcc_path(), *NVCC_FLAGS, "-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
        print(" ".join(cmd))
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed building libdescribealign_b200.so")
    if verbose:
        print(res.stdout + res.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
