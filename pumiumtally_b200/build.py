"""In-tree build of libpumitally.so (CUDA kernels + C++ host side + C ABI).

``nvcc`` cross-compiles for sm_100a without a GPU, so this runs in the CPU
container; the resulting ``pumiumtally_b200/lib/libpumitally.so`` travels to
the GPU box with the repo snapshot (it is git-ignored, not gpurun-ignored).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIBDIR = os.path.join(PKG, "lib")
OBJDIR = os.path.join(PKG, "build")
LIB = os.path.join(LIBDIR, "libpumitally.so")
LIB_EXP = os.path.join(LIBDIR, "libpumitally_exp.so")  # product + measured alternatives (tests/experiments only)

SOURCES = [
    "walk_kernels.cu",
    "bin_kernels.cu",
    "batch_stats.cu",
    "engine.cu",
    "host_stage.cpp",
    "tet_mesh.cpp",
    "osh_reader.cpp",
    "gmsh_reader.cpp",
    "vtk_writer.cpp",
    "nccl_dl.cpp",
    "c_api.cpp",
    "pumitally_facade.cpp",
]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-fopenmp,-pthread,-Wall,-fvisibility=default",
    "-I", os.path.join(ROOT, "include"),
    "-I", CSRC,
]


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libpumitally.so cannot be built")


def _newer(a: str, b: str) -> bool:
    return (not os.path.exists(b)) or os.path.getmtime(a) > os.path.getmtime(b)


def build_library(force: bool = False, verbose: bool = False, experiments: bool = False) -> str:
    """Compile every translation unit that changed and relink. Returns the .so path.

    experiments=True builds lib/libpumitally_exp.so instead: the same library plus the measured
    alternative kernels of csrc/experiments/ (flag PTB_EXPERIMENTS); select it at run time with
    PUMITALLY_LIB=<path>.  The product library never contains them."""
    os.makedirs(LIBDIR, exist_ok=True)
    objdir = OBJDIR + ("_exp" if experiments else "")
    os.makedirs(objdir, exist_ok=True)
    lib = LIB_EXP if experiments else LIB
    sources = SOURCES + (["experiments/walk_experiments.cu"] if experiments else [])
    flags = NVCC_FLAGS + (["-DPTB_EXPERIMENTS"] if experiments else [])
    nvcc = _nvcc()
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".hpp", ".cuh", ".h"))]
    headers += [os.path.join(ROOT, "include", "pumitally_c.h"),
                os.path.join(ROOT, "include", "pumitally", "PumiTally.h")]
    newest_header = max(os.path.getmtime(h) for h in headers)
    objs, relink = [], force or not os.path.exists(lib)
    for src in sources:
        s = os.path.join(CSRC, src)
        o = os.path.join(objdir, src.replace("/", "_") + ".o")
        objs.append(o)
        if force or _newer(s, o) or newest_header > os.path.getmtime(o):
            cmd = [nvcc, *flags, "-c", s, "-o", o]
            if verbose:
                print(" ".join(cmd), file=sys.stderr)
            subprocess.check_call(cmd)
            relink = True
    if relink:
        cmd = [nvcc, "-shared", "-o", lib, *objs, "-Xcompiler", "-fopenmp,-pthread", "-lgomp", "-ldl", "-lz",
               "-gencode", "arch=compute_100a,code=sm_100a"]
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        subprocess.check_call(cmd)
    return lib


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose=True, experiments="--experiments" in sys.argv))
