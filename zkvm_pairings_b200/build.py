"""Builds libzkpair.so (hand-written CUDA for sm_100a + the C ABI of include/zkpair.h) in-tree.

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box with the
snapshot.  Usage: python -m zkvm_pairings_b200.build [--force] [-DNAME=VALUE ...]
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libzkpair.so")
SOURCES = ["kernels.cu", "pairing_kernel.cu", "fe_kernel.cu"]
HEADERS = ["fp.cuh", "tower.cuh", "pairing.cuh", "ops.cuh", "fe_scratch.cuh", "groth16.cuh", "kzg.cuh", "fr.cuh", "blob.cuh", "kzg_prove.cuh", "kzg_cells.cuh", "kzg_recover.cuh", "msm.cuh", "consts.cuh", "../../include/zkpair.h"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared", "--threads", "0"]   # the three units compile in parallel


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (needed to build libzkpair.so for sm_100a)")


def is_stale(so: str = SO) -> bool:
    if not os.path.exists(so):
        return True
    t = os.path.getmtime(so)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, defines=(), out: str = SO, verbose: bool = False) -> str:
    consts = os.path.join(CSRC, "consts.cuh")
    if not os.path.exists(consts):
        subprocess.check_call([sys.executable, os.path.join(CSRC, "gen_consts.py")])
    if not force and not is_stale(out):
        return out
    cmd = [nvcc_path()] + NVCC_FLAGS + list(defines) + (["-Xptxas", "-v"] if verbose else []) + \
        ["-o", out] + [os.path.join(CSRC, s) for s in SOURCES]
    subprocess.check_call(cmd, cwd=CSRC)
    return out


if __name__ == "__main__":
    defs = [a for a in sys.argv[1:] if a.startswith("-D")]
    print(build(force="--force" in sys.argv, defines=defs, verbose="-v" in sys.argv))
