"""Builds libgnan_b200.so (the C-ABI library of include/gnan_b200.h) in-tree with nvcc for sm_100a.

    python graph-neural-additive-networks---gnan_b200/build.py [--force]

nvcc cross-compiles without a GPU. Objects go to csrc/_build/, the shared library next to this file so that
it travels with the repo snapshot (it is git-ignored).
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "_build")
LIB = os.path.join(HERE, "libgnan_b200.so")
SOURCES = ["api.cu", "mlp.cu", "mlp_tc.cu", "agg.cu", "agg_tc.cu", "agg_bd.cu", "apsp.cu", "csr.cu", "entries.cu", "train.cu", "wide.cu", "explain.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-I" + os.path.join(ROOT, "include"), "-Xcompiler", "-fPIC"]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(ROOT, "include", "gnan_b200.h"))

    def compile_one(src):
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src[:-3] + ".o")
        if force or _stale(o, [s] + headers):
            cmd = [NVCC] + FLAGS + ["-c", s, "-o", o]
            if verbose:
                print(" ".join(cmd), flush=True)
            subprocess.check_call(cmd)
            return o, True
        return o, False

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        res = list(ex.map(compile_one, SOURCES))
    objs = [o for o, _ in res]
    if force or any(c for _, c in res) or _stale(LIB, objs):
        cmd = [NVCC, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "shared"]
        if verbose:
            print(" ".join(cmd), flush=True)
        subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
