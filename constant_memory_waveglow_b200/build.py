"""Build libcmwg_b200.so (sm_100a only) with nvcc, in-tree.

    python -m constant_memory_waveglow_b200.build [--force]

The shared library is written to constant_memory_waveglow_b200/lib/ (git-ignored, shipped to the
GPU box with the repo snapshot).  nvcc cross-compiles without a GPU.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
OBJDIR = os.path.join(LIBDIR, "obj")
LIB = os.path.join(LIBDIR, "libcmwg_b200.so")
SOURCES = ["flow_elementwise.cu", "upsample.cu", "melspec.cu", "denoise.cu", "waveflow.cu", "wsrglow_cond.cu", "lvc.cu",
           "engine_tc.cu", "wn_pipeline.cu", "nvidia_upsample.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _deps_mtime() -> float:
    m = 0.0
    for root in (CSRC, os.path.join(os.path.dirname(HERE), "include")):
        for f in os.listdir(root):
            if f.endswith((".cu", ".cuh", ".h")):
                m = max(m, os.path.getmtime(os.path.join(root, f)))
    return max(m, os.path.getmtime(os.path.abspath(__file__)))


def needs_build() -> bool:
    return not os.path.exists(LIB) or os.path.getmtime(LIB) < _deps_mtime()


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    os.makedirs(OBJDIR, exist_ok=True)
    nvcc = _nvcc()

    def compile_one(src: str) -> str:
        obj = os.path.join(OBJDIR, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas")
            cmd.insert(2, "-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    tmp = LIB + ".tmp"
    r = subprocess.run([nvcc, "-shared", "-o", tmp, *objs, "-gencode", "arch=compute_100a,code=sm_100a"],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    os.replace(tmp, LIB)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
