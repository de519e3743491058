"""Build libpde_b200.so in-tree with nvcc for sm_100a (no torch headers, plain C ABI).

    python cnn-with-pde_b200/build.py [--force] [--verbose]

nvcc cross-compiles without a GPU; the .so is git-ignored but travels with the gpurun snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(ROOT, "include")
LIB = os.path.join(HERE, "libpde_b200.so")
SOURCES = ["cabi.cu", "adi.cu", "adi_split.cu", "adi_generic.cu", "adi_wide.cu", "explicit.cu", "tiny_split.cu", "tiny_tiled.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
    # IEEE arithmetic on purpose: no --use_fast_math, no flush-to-zero (SVHN's default
    # channel_coupling = 0.01 I drives the field to ~1e-20, SURVEY.md appendix B.7)
    "--ftz=false", "--prec-div=true", "--prec-sqrt=true",
    "-I", INCLUDE, "-I", CSRC,
]


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libpde_b200.so cannot be built (there is no CPU fallback)")


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(INCLUDE, "pde_b200.h"), __file__]
    return any(os.path.getmtime(p) > t for p in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    nvcc = _nvcc()
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    env = dict(os.environ)
    # the image exports CC/CXX wrappers that break host compilation; use the system g++
    ccbin = shutil.which("g++") or "/usr/bin/g++"

    extra = os.environ.get("PDE_B200_NVCC_EXTRA", "").split()   # e.g. -DPDE_BWD_MINBLOCKS=1 for A/B builds

    def compile_one(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc, "-ccbin", ccbin] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + \
              ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, env=env, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, "-ccbin", ccbin, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs + \
          ["-lcudart_static", "-lrt", "-ldl", "-lpthread"]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
