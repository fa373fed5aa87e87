"""Build recipe of libamira_gmg.so: plain nvcc, sm_100a only, in-tree (the .so travels with the
repository snapshot to the GPU box; it is git-ignored)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libamira_gmg.so")
SOURCES = ["gmg.cu", "comm.cu", "vocab_encode.cpp", "host_keys.cpp"]
HEADERS = ["common.cuh", "gmg_kernels.cuh", "post_kernels.cuh", "scan.cuh", "segsort.cuh", "incidence.cuh", "stats.cuh", "paths.cuh", "unitigs.cuh", "bubbles.cuh", "correct.cuh", "tips.cuh", "gene_paths.cuh", "sharded.cuh", os.path.join("..", "..", "include", "amira_gmg.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "--use_fast_math",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall", "-shared"]


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    extra = os.environ.get("AMIRA_NVCC_FLAGS", "").split()       # developer experiments (e.g. -DAMIRA_INS_ILP=1)
    out = os.environ.get("AMIRA_LIB_OUT", LIB)
    cmd = [NVCC] + FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-o", out] + \
          [os.path.join(CSRC, f) for f in SOURCES] + ["-lcudart", "-lpthread"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed building libamira_gmg.so")
    if verbose:
        sys.stderr.write(res.stdout + res.stderr)
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
