"""Builds libspliser_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libspliser_b200.so")
SOURCES = ["kernels.cu", "count_fused.cu", "graph_build.cu", "bam_gpu.cu", "strand_votes.cu", "group_split.cu", "pipeline.cu", "site_graph.cpp", "bam_io.cpp", "host_text.cpp"]
HEADERS = ["device_types.h", "dev_helpers.cuh", "graph_build.h", "bam_gpu.h", "inflate.h", "site_graph.h", "bam_io.h", "bam_aux.h", "read_filter.h", "junction_filter.h", "strand_votes.h", "tag_groups.h", "group_split.h", os.path.join("..", "..", "include", "spliser_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC,-Wall", "-shared"]


def _nvcc() -> str:
    cand = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(cand):
        raise RuntimeError("nvcc not found; libspliser_b200.so cannot be built")
    return cand


def is_stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB
    extra = os.environ.get("SPLISER_NVCC_FLAGS", "").split()      # tuning experiments only (e.g. -DSPL_K3_DENSE=8)
    cmd = [_nvcc()] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + SOURCES + ["-lz"]
    res = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n%s\n%s" % (res.stdout, res.stderr))
    if verbose:
        sys.stderr.write(res.stderr)
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
