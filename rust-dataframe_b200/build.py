"""Builds rust-dataframe_b200/libb200df.so from csrc/*.cu with nvcc for sm_100a (cross-compiles without a GPU).

The shared library is the product: a C-ABI (include/b200df.h) over hand-written CUDA kernels.  It is built
in-tree so that it travels with the repository snapshot to the GPU box.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
ROOT = os.path.dirname(HERE)
LIB = os.path.join(HERE, "libb200df.so")
OBJ_DIR = os.path.join(HERE, "build")
SOURCES = ["k_binary.cu", "k_unary.cu", "k_cast.cu", "k_reduce.cu", "k_filter.cu", "k_expr.cu", "k_sort.cu", "k_group.cu", "k_generate.cu", "runtime.cu", "fleet.cu", "ipc.cu", "comm.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _deps_mtime() -> float:
    paths = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(ROOT, "include", "b200df.h"), __file__]
    return max(os.path.getmtime(p) for p in paths)


def needs_build() -> bool:
    return not os.path.exists(LIB) or os.path.getmtime(LIB) < _deps_mtime()


def build_native(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    os.makedirs(OBJ_DIR, exist_ok=True)
    nvcc = _nvcc()
    hdr_mtime = max(os.path.getmtime(os.path.join(CSRC, "common.cuh")), os.path.getmtime(os.path.join(CSRC, "comm.cuh")),
                    os.path.getmtime(os.path.join(CSRC, "runtime.cuh")), os.path.getmtime(os.path.join(ROOT, "include", "b200df.h")),
                    os.path.getmtime(__file__))

    def compile_one(src: str) -> str:
        obj = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        srcp = os.path.join(CSRC, src)
        if not force and os.path.exists(obj) and os.path.getmtime(obj) >= max(os.path.getmtime(srcp), hdr_mtime):
            return obj
        cmd = [nvcc] + NVCC_FLAGS + ["-c", srcp, "-o", obj]
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC", "-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    print(build_native(force="--force" in sys.argv, verbose=True))
