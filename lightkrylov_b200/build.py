"""Build liblkb.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python -m lightkrylov_b200.build [--force]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(CSRC, "liblkb.so")
SOURCES = ["kernels_gs.cu", "kernels_vec.cu", "kernels_ops.cu", "kernels_gemm.cu", "kernels_fused.cu", "lkb_core.cu", "lkb_cheb.cu", "lkb_poly.cu", "lkb_mg.cu", "lkb_csr.cu", "lkb_krylov.cu",
           "lkb_solvers.cu", "lkb_eig.cu", "lkb_expm.cu"]
# every header in csrc/ (globbed: a forgotten header once left objects stale) + the public C ABI
HEADERS = sorted(f for f in os.listdir(CSRC) if f.endswith((".h", ".cuh", ".inc"))) + [os.path.join("..", "..", "include", "lkb.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=default", "-ccbin", "/usr/bin/g++"]


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    objdir = os.path.join(CSRC, "build")
    os.makedirs(objdir, exist_ok=True)

    def compile_one(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        if force or _stale(obj, [os.path.join(CSRC, src)] + hdrs):
            cmd = [NVCC] + FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
            if verbose:
                print(" ".join(cmd))
            subprocess.check_call(cmd)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        objs = list(ex.map(compile_one, srcs))
    if force or _stale(OUT, objs):
        cmd = [NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", OUT] + objs + \
              ["-cudart", "static", "-ldl", "-lpthread", "-ccbin", "/usr/bin/g++"]
        if verbose:
            print(" ".join(cmd))
        subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
