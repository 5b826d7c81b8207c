"""Build libihtb200.so (sm_100a only) in-tree with nvcc.  No GPU is needed to build."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libihtb200.so")
SOURCES = ["geno.cu", "dense.cu", "bgen.cu", "support.cu", "sweep.cu", "sweep_lut.cu", "sweep_tmem.cu", "sweep_lut64.cu", "glm.cu", "topk.cu", "fit.cu", "comm.cu", "mvfit.cu", "p2p.cu", "debias.cu", "groups.cu", "multi.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-fmad=false", "-std=c++17",
              "-Xcompiler", "-fPIC"]


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libihtb200.so cannot be built")


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    nvcc = _nvcc()
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(HERE, "..", "include", "ihtb200.h"))

    def compile_one(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        path = os.path.join(CSRC, src)
        if force or _stale(obj, [path] + headers):
            cmd = [nvcc] + NVCC_FLAGS + ["-c", path, "-o", obj]
            if verbose:
                print(" ".join(cmd), file=sys.stderr)
            subprocess.run(cmd, check=True)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    if force or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs + ["-ldl"]
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
