"""Builds permon_b200/libpermon_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m permon_b200.build [--force]

The library is the product: CUDA kernels + the C ABI declared in include/permon_b200.h.  It links the CUDA
runtime statically and NCCL dynamically (libnccl.so.2; the copy torch already loaded is reused).
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "csrc", "build")
LIB = os.path.join(HERE, "libpermon_b200.so")
SOURCES = ["kernels.cu", "shim.cpp", "qp.cpp", "qps.cpp", "pack.cpp", "qps_lin.cpp", "recode.cu"]
HEADERS = ["device.h", "mpgp_ctl.h", "objects.h", os.path.join("..", "..", "include", "permon_b200.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-std=c++17", "-O3", "-lineinfo", "--extended-lambda", "-Xcompiler", "-fPIC,-fvisibility=hidden,-Wall,-Wno-maybe-uninitialized,-fopenmp",
          "-ccbin", "/usr/bin/g++"]


def _newer(src, dst):
    return not os.path.exists(dst) or os.path.getmtime(src) > os.path.getmtime(dst)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    hdr_paths = [os.path.join(CSRC, h) for h in HEADERS]
    objs = []
    relink = force or not os.path.exists(LIB)
    todo = []
    for src in SOURCES:
        sp = os.path.join(CSRC, src)
        op = os.path.join(OBJ, src.rsplit(".", 1)[0] + ".o")
        objs.append(op)
        if force or _newer(sp, op) or any(_newer(h, op) for h in hdr_paths):
            todo.append([NVCC, *ARCH, *COMMON, "-x", "cu", "-c", sp, "-o", op])
    if todo:   # the translation units are independent: compile them side by side (kernels.cu dominates)
        from concurrent.futures import ThreadPoolExecutor

        def run(cmd):
            if verbose:
                print(" ".join(cmd), flush=True)
            subprocess.check_call(cmd)

        with ThreadPoolExecutor(max_workers=min(len(todo), os.cpu_count() or 1)) as ex:
            list(ex.map(run, todo))
        relink = True
    if relink:
        cmd = [NVCC, *ARCH, "-shared", "-ccbin", "/usr/bin/g++", "-o", LIB, *objs, "-lnccl", "-lgomp", "-Xlinker", "--no-undefined"]
        if verbose:
            print(" ".join(cmd), flush=True)
        subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
