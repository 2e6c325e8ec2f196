"""Builds libtfrecomm.so (hand-written sm_100a CUDA + the C ABI of include/tfrecomm.h) IN-TREE with nvcc.

nvcc cross-compiles without a GPU; the .so is git-ignored but travels to the GPU box with the snapshot.
cudart is linked statically (nvcc default) so the library does not depend on which libcudart torch ships.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "_obj")
SO = os.path.join(HERE, os.environ.get("TFR_SO_NAME", "libtfrecomm.so"))
OBJ = OBJ + os.environ.get("TFR_OBJ_SUFFIX", "")
SOURCES = ["svd_forward.cu", "dedup_sort.cu", "segsum.cu", "adam.cu", "adam_ring.cu", "fm.cu", "shard.cu", "allpairs.cu", "metrics.cu", "rank_users.cu", "fold_in.cu", "capi.cu"]
NVCC = os.environ.get("TFR_NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
         "-ccbin", "/usr/bin/g++", "-Xcompiler", "-fPIC,-fopenmp"] + os.environ.get("TFR_EXTRA_NVCC_FLAGS", "").split()


def _deps_mtime():
    inc = os.path.join(HERE, "..", "include", "tfrecomm.h")
    return max(os.path.getmtime(p) for p in [inc] + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")])


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    dep = _deps_mtime()
    todo = []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        obj = os.path.join(OBJ, s[:-3] + ".o")
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), dep):
            todo.append((src, obj))

    def cc(so):
        cmd = [NVCC] + FLAGS + ["-c", so[0], "-o", so[1]]
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        subprocess.check_call(cmd)

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(todo)))) as ex:
        list(ex.map(cc, todo))
    objs = [os.path.join(OBJ, s[:-3] + ".o") for s in SOURCES]
    if todo or not os.path.exists(SO):
        # -fopenmp: the host-side feed packing (tfr_host_pack_feed) splits a batch over a few threads
        subprocess.check_call([NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-ccbin", "/usr/bin/g++",
                               "-Xcompiler", "-fopenmp", "-o", SO] + objs)
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
