"""Builds libii2.so (CUDA, sm_100a only) in-tree with nvcc.

The library is a plain C-ABI shared object (include/ii2.h) with no torch dependency, so
the Go host can bind it through cgo exactly as the Python tests bind it through ctypes.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libii2.so")
SOURCES = ["runtime.cu", "k3a_intcomp.cu", "k1_plan.cu", "k12_union.cu", "k12_fused.cu", "k6_emit.cu",
           "k5_prefix.cu", "k7_ingest.cu", "k8_lookup.cu", "k9_query.cu", "k10_pattern.cu", "k3b_bitmask.cu", "api.cu", "comm.cu", "fst_v1.cpp", "removed_gob.cpp"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC"]


def _newer(srcs, target):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in srcs)


def build(force: bool = False, verbose: bool = False) -> str:
    nvcc = os.environ.get("NVCC", "nvcc")
    if not os.path.isdir(CSRC):
        if os.path.exists(OUT):
            return OUT
        raise RuntimeError("no CUDA sources and no prebuilt libii2.so")
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hdrs.append(os.path.join(HERE, "..", "include", "ii2.h"))
    srcs = [os.path.join(CSRC, f) for f in SOURCES]
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)

    def compile_one(src):
        obj = os.path.join(objdir, os.path.splitext(os.path.basename(src))[0] + ".o")
        if force or _newer([src] + hdrs, obj):
            cmd = [nvcc] + NVCC_FLAGS + ["-c", src, "-o", obj]
            if verbose:
                print(" ".join(cmd), file=sys.stderr)
            subprocess.check_call(cmd)
        return obj

    with ThreadPoolExecutor(max_workers=8) as ex:
        objs = list(ex.map(compile_one, srcs))
    if force or _newer(objs, OUT):
        cmd = [nvcc, "-shared", "-o", OUT] + objs + ["-gencode", "arch=compute_100a,code=sm_100a",
                                                     "-cudart", "shared", "-ldl"]
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
