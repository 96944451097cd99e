"""Build csrc/libedgcn.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(CSRC, "libedgcn.so")
SOURCES = ["libedgcn.cu", "edg_api.cu", "edg_graph.cu", "edg_aggregate.cu", "edg_gemm_simt.cu", "edg_gemm_tc.cu", "edg_split.cu",
           "edg_block.cu", "edg_block_staged.cu", "edg_pairs.cu", "edg_staged.cuh", "edg_block_head.cu", "edg_loss.cu", "edg_segment.cu", "edg_optim.cu", "edg_mlp_chain.cu", "edg_gcn_fused.cu", "edg_head_fused.cu", "edg_common.cuh", os.path.join("..", "..", "include", "edgcn.h")]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def stale() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(os.path.join(CSRC, s)) > t for s in SOURCES)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not stale():
        return OUT
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", OUT, "libedgcn.cu"]
    r = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed building libedgcn.so")
    if verbose:
        print(r.stderr)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
