"""Build recipes: the CUDA C-ABI library (sm_100a only) and the C++ host executable.

Everything is built IN-TREE (xalm_b200/libxalm_cuda.so, xalm_b200/xalm_main) so the artefacts travel to the
GPU box with the repo snapshot.  nvcc cross-compiles without a GPU.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libxalm_cuda.so")
MAIN = os.path.join(HERE, "xalm_main")
HOSTLIB = os.path.join(HERE, "libxalm_host.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
GXX = "/usr/bin/g++"   # the image's $CXX points at a wrapper without OpenMP specs; name the system compiler

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--use_fast_math=false",
              "-Xcompiler", "-fPIC", "-ccbin", GXX]
NVCC_FLAGS = [f for f in NVCC_FLAGS if f != "--use_fast_math=false"]


def _newer(target: str, sources) -> bool:
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(s) <= t for s in sources)


def _sources(d, exts):
    out = []
    for base, _, files in os.walk(d):
        for f in files:
            if f.endswith(exts):
                out.append(os.path.join(base, f))
    return out


CUDA_TUS = ["xalm_cuda.cu", "prefill.cu"]   # translation units of libxalm_cuda.so (objects cached under csrc/.obj)


def build_cuda(force: bool = False, verbose: bool = False, extra=()) -> str:
    hdrs = _sources(CSRC, (".cuh", ".h")) + [os.path.join(ROOT, "include", "xalm_cuda.h")]
    hdrs = [h for h in hdrs if os.sep + "host" + os.sep not in h]
    objdir = os.path.join(CSRC, ".obj")
    os.makedirs(objdir, exist_ok=True)
    objs, procs = [], []
    for tu in CUDA_TUS:
        src = os.path.join(CSRC, tu)
        obj = os.path.join(objdir, tu.replace(".cu", ".o"))
        objs.append(obj)
        if not force and not extra and _newer(obj, [src] + hdrs):
            continue
        cmd = [NVCC, *NVCC_FLAGS, *extra, "-c", "-o", obj, src]
        if verbose:
            cmd[1:1] = ["-Xptxas", "-v"]
            print(" ".join(cmd))
        procs.append((cmd, subprocess.Popen(cmd)))
    for cmd, p in procs:
        if p.wait() != 0:
            raise subprocess.CalledProcessError(p.returncode, cmd)
    if procs or not os.path.exists(LIB) or not _newer(LIB, objs):
        subprocess.check_call([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB, *objs, "-ldl", "-ccbin", GXX])
    return LIB


def build_host(force: bool = False) -> str:
    """libxalm_host.so: format writers + synthetic generator (no CUDA dependency, loaded by synth.py).
    xalm_main: the C++ host executable (reference CLI surface) linked against libxalm_cuda.so."""
    hdir = os.path.join(CSRC, "host")
    deps = _sources(hdir, (".cpp", ".h")) + [os.path.join(ROOT, "include", "xalm_cuda.h")]
    common = [GXX, "-O2", "-std=c++20", "-fPIC", "-fopenmp", "-Wall", "-I", os.path.join(ROOT, "include"), "-I", hdir]
    quant = os.path.join(hdir, "quantize.cpp")
    if force or not _newer(HOSTLIB, [quant]):
        subprocess.check_call([*common, "-shared", "-o", HOSTLIB, quant])
    main_src = os.path.join(hdir, "main.cpp")
    if os.path.exists(main_src) and (force or not _newer(MAIN, deps + [LIB])):
        build_cuda()
        subprocess.check_call([*common, "-o", MAIN, main_src, os.path.join(hdir, "launch.cpp"), os.path.join(hdir, "model.cpp"), quant, "-L", HERE, "-lxalm_cuda",
                               "-Wl,-rpath,$ORIGIN"])
    return HOSTLIB


def build_all(force: bool = False, verbose: bool = False):
    build_cuda(force, verbose)
    build_host(force)


if __name__ == "__main__":
    build_all(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print("built", LIB)
