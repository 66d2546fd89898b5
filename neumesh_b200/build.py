"""Build ``libneumesh_b200.so`` (hand-written sm_100a CUDA behind a C ABI) and the oracle's C helpers, in-tree.

``python -m neumesh_b200.build`` or ``__graft_entry__.build()``.  nvcc cross-compiles without a GPU.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libneumesh_b200.so")
SOURCES = ["api.cu", "grid.cu", "field.cu", "field_ffma.cu", "field_tc.cu", "render.cu", "shell.cu", "train.cu",
           "mcubes.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
              "--expt-relaxed-constexpr"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _newer(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(LIB_DIR, exist_ok=True)
    obj_dir = os.path.join(HERE, "build")
    os.makedirs(obj_dir, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "neumesh_b200.h"))
    nvcc = _nvcc()

    def compile_one(src):
        obj = os.path.join(obj_dir, src.replace(".cu", ".o"))
        path = os.path.join(CSRC, src)
        if force or _newer(obj, [path] + headers):
            cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", path, "-o", obj]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
            if verbose:
                print(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    if force or _newer(LIB_PATH, objs):
        cmd = [nvcc, "-shared", "-o", LIB_PATH] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
