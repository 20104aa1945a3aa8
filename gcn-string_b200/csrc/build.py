"""Compile the C-ABI CUDA library in-tree with plain nvcc for sm_100a.

    python gcn-string_b200/csrc/build.py [--force] [--verbose]

Output: gcn-string_b200/libgcnstring_b200.so (git-ignored; it travels to the GPU box with
the gpurun snapshot).  Objects are cached under gcn-string_b200/csrc/build/ and rebuilt
only when a source or header is newer.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(HERE)
ROOT = os.path.dirname(PKG)
OUT = os.path.join(PKG, "libgcnstring_b200.so")
OBJ = os.path.join(HERE, "build")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
SOURCES = ["api.cu", "batching.cu", "spmm.cu", "spmm_slab.cu", "linear.cu", "linear_tc.cu", "bn.cu", "pool.cu", "pool_attn.cu", "loss.cu", "optim.cu", "model.cu", "attr.cu", "contact.cu", "comm.cu"]
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
         "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]


def _headers():
    hs = [os.path.join(HERE, f) for f in os.listdir(HERE) if f.endswith((".cuh", ".h"))]
    hs.append(os.path.join(ROOT, "include", "gcnstring_b200.h"))
    return hs


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    hdrs = _headers() + [os.path.abspath(__file__)]
    extra = ["-Xptxas", "-v"] if verbose else []

    def compile_one(src):
        s = os.path.join(HERE, src)
        o = os.path.join(OBJ, src.replace(".cu", ".o"))
        if force or _stale(o, [s] + hdrs):
            cmd = [NVCC] + FLAGS + extra + ["-c", s, "-o", o]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
            if verbose:
                sys.stderr.write(r.stderr)
        return o

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    if force or _stale(OUT, objs):
        cmd = [NVCC, "-shared", "-o", OUT] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart_static", "-ldl", "-lrt", "-lpthread"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
