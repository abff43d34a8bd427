"""Build libskani_b200.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "_lib")
LIB = os.path.join(LIBDIR, "libskani_b200.so")
SOURCES = ["skb_api.cu", "fasta_pack.cpp"]
HEADERS = ["skb_common.cuh", "skb_sketch.cuh", "skb_index.cuh", "skb_probe.cuh", "skb_ani.cuh", "skb_best_n.cuh", "skb_matrix.cuh", "skb_table_blocks.cuh", "../../include/skani_b200.h"]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def build(force=False, verbose=False):
    if not force and not _stale():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [
        nvcc, "-O3", "-std=c++17",
        "-gencode", "arch=compute_100a,code=sm_100a",
        "-lineinfo", "-Xcompiler", "-fPIC", "-shared",
        "-o", LIB,
    ] + [os.path.join(CSRC, s) for s in SOURCES] + ["-lz"]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
        print(" ".join(cmd), file=sys.stderr)
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
