"""Builds libswb200.so (+ libswb200.a) in-tree with nvcc for sm_100a.

    python -m simpleworks_b200.build [--force]

The shared object is what the ctypes loader and the tests use; the static archive is what a Rust
build.rs would link (see INTEGRATION.md).  Both are git-ignored build artefacts that travel to the
GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
BUILD = os.path.join(HERE, "_build")
SOURCES = ["ctx.cu", "vec.cu", "ntt.cu", "msm.cu", "msm_sort.cu", "radix_sort.cu", "msm_accumulate.cu", "msm_pairs.cu", "msm_reduce.cu", "fixed_base.cu", "polyops.cu", "marlin_ops.cu",
           "marlin_abi.cu", "comm.cu", "index_ops.cu", "verify_ops.cu"]
LIB_SO = os.path.join(HERE, "libswb200.so")
LIB_A = os.path.join(HERE, "libswb200.a")
NVCC = os.environ.get("SWB_NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
         "-Xcompiler", "-fPIC,-fopenmp", "--expt-relaxed-constexpr", "-ccbin", "/usr/bin/g++"]


def _deps():
    out = []
    for root, _, files in os.walk(CSRC):
        out += [os.path.join(root, f) for f in files]
    out.append(os.path.join(HERE, "..", "include", "swb200.h"))
    return out


def needs_build() -> bool:
    if not (os.path.exists(LIB_SO) and os.path.exists(LIB_A)):
        return True
    t = min(os.path.getmtime(LIB_SO), os.path.getmtime(LIB_A))
    return any(os.path.getmtime(d) > t for d in _deps())


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB_SO
    os.makedirs(BUILD, exist_ok=True)
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]

    def compile_one(src):
        obj = os.path.join(BUILD, src.replace(".cu", ".o"))
        cmd = [NVCC, *FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            print(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(srcs)) as ex:
        objs = list(ex.map(compile_one, srcs))
    r = subprocess.run([NVCC, "-shared", "-o", LIB_SO, *objs, "-lcudart_static", "-ldl", "-lrt", "-lpthread", "-lgomp"],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    if os.path.exists(LIB_A):
        os.remove(LIB_A)
    subprocess.check_call(["ar", "rcs", LIB_A, *objs])
    return LIB_SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
