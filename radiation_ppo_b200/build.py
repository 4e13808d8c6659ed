"""Builds radiation_ppo_b200/_C/libradsearch_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

`python -m radiation_ppo_b200.build [--force]`.  nvcc cross-compiles without a GPU; the .so is git-ignored but travels
to the GPU box with the tree.  -fmad=false: the fp64 arithmetic that must match numpy / scipy bit for bit (Poisson PTRS,
GAE recurrence, reward rounding) must not be contracted into fused multiply-adds.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC_DIR = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "_C")
LIB = os.path.join(OUT_DIR, "libradsearch_b200.so")
SOURCES = ["rs_kernels.cu", "rs_gae.cu", "rs_maps.cu", "rs_pack.cu", "rs_rollout.cu", "rs_eval.cu", "rs_policy.cu"]
NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-fmad=false",
    "-Xcompiler", "-fPIC", "-shared", "-cudart", "static",
]


def _newest_source_mtime() -> float:
    m = 0.0
    for root in (SRC_DIR, os.path.join(HERE, "..", "include")):
        for f in os.listdir(root):
            m = max(m, os.path.getmtime(os.path.join(root, f)))
    return m


def build(force: bool = False, verbose: bool = False, defines=(), out: str = LIB) -> str:
    """defines / out: a variant build with -D tuning macros (e.g. RS_STEP1_OCC=8) written next to the shipped library;
    load it with RADSEARCH_B200_LIB=<path> (measurement only: tools/gpu_variants.sh)."""
    os.makedirs(os.path.dirname(out), exist_ok=True)
    if not force and os.path.exists(out) and os.path.getmtime(out) >= _newest_source_mtime():
        return out
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc, *NVCC_FLAGS, *( ["-Xptxas", "-v"] if verbose else []), *[f"-D{d}" for d in defines], "-o", out,
           *[os.path.join(SRC_DIR, s) for s in SOURCES]]
    subprocess.run(cmd, check=True)
    return out


if __name__ == "__main__":
    defs = [a[2:] for a in sys.argv[1:] if a.startswith("-D")]
    outs = [a[2:] for a in sys.argv[1:] if a.startswith("-o")]
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, defines=defs,
                out=os.path.join(OUT_DIR, outs[0]) if outs else LIB))
