"""Build libcbo_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m cbo_with_oop_b200.build [--force] [--verbose]

The shared object is written next to this file so that it travels with the repository snapshot to the GPU
box; it is git-ignored.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(HERE, "..", "include")
LIB = os.path.join(HERE, "libcbo_b200.so")
SOURCES = ["api.cu", "tables.cu", "prior_precompute.cu", "prior_eval.cu", "prior_pair.cu", "prior_rows.cu", "posterior_fit.cu", "sweep.cu", "obs_gp_fit.cu", "sem.cu", "refine.cu", "posterior_hyper.cu"]
HEADERS = ["cbo_common.cuh", "dmma_tile.cuh", "dmma_tma_tile.cuh", "m_triangle_pass.cuh", "prior_pair.cuh", "surrogate.cuh", os.path.join(INCLUDE, "cbo_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + [h if os.path.isabs(h) else os.path.join(CSRC, h) for h in HEADERS]
    deps.append(os.path.abspath(__file__))
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force: bool = False, verbose: bool = False) -> str:
    """Compile every CUDA translation unit and link the C-ABI shared library.  Returns its path."""
    if not force and not _stale():
        return LIB
    nvcc = _nvcc()
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    extra = ["-Xptxas", "-v"] if verbose else []
    extra += os.environ.get("CBO_NVCC_EXTRA", "").split()

    def compile_one(src: str) -> str:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, *extra, "-I", INCLUDE, "-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
