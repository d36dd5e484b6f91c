"""Build librip_cuda.so (CUDA kernels + C ABI) and librip_host.so (C++ host classes) in-tree.

    python opencl-development-real-time-image-processing_b200/build.py [--force] [--verbose]

nvcc cross-compiles for sm_100a without a GPU; the built .so files are git-ignored but travel to
the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import argparse
import glob
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
HOST = os.path.join(PKG, "host")
INCLUDE = os.path.join(ROOT, "include")
LIB_CUDA = os.path.join(PKG, "librip_cuda.so")
LIB_HOST = os.path.join(PKG, "librip_host.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "--shared", "-Xcompiler", "-fPIC,-ffp-contract=off,-Wall", "-Xptxas", "-v",
    "-I", INCLUDE, "-I", CSRC, "-cudart", "shared",
]


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found: librip_cuda.so cannot be built (there is no CPU fallback)")


def _host_cxx() -> str:
    # the image exports CXX=/opt/gcc/bin/g++ without libgomp/specs; prefer the system compiler
    for c in ("/usr/bin/g++", shutil.which("g++")):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("g++ not found")


def _stale(target: str, sources: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def build_cuda(force: bool = False, verbose: bool = False) -> str:
    srcs = sorted(glob.glob(os.path.join(CSRC, "*.cu")))
    deps = srcs + glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(CSRC, "*.h")) + \
        glob.glob(os.path.join(INCLUDE, "*.h"))
    if force or _stale(LIB_CUDA, deps):
        extra = os.environ.get("RIP_NVCC_DEFS", "").split()
        cmd = [_nvcc(), *NVCC_FLAGS, *extra, "-ccbin", _host_cxx(), "-o", os.environ.get("RIP_LIB_OUT", LIB_CUDA), *srcs]
        res = subprocess.run(cmd, capture_output=True, text=True)
        log = res.stdout + res.stderr
        with open(os.path.join(PKG, "build_cuda.log"), "w") as f:
            f.write(" ".join(cmd) + "\n" + log)
        if verbose or res.returncode:
            sys.stderr.write(log)
        if res.returncode:
            raise RuntimeError("nvcc failed building librip_cuda.so (see build_cuda.log)")
    return LIB_CUDA


def build_host(force: bool = False, verbose: bool = False) -> str | None:
    srcs = sorted(glob.glob(os.path.join(HOST, "*.cpp")))
    if not srcs:
        return None
    deps = srcs + glob.glob(os.path.join(HOST, "*.hpp")) + glob.glob(os.path.join(HOST, "*.h")) + \
        glob.glob(os.path.join(INCLUDE, "*.h")) + [os.path.join(CSRC, "rip_formats.h")]
    if force or _stale(LIB_HOST, deps) or _stale(LIB_HOST, [LIB_CUDA]):
        cmd = [_host_cxx(), "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-Wall", "-pthread",
               "-I", INCLUDE, "-I", HOST, "-I", CSRC, "-I", os.path.join(os.path.dirname(os.path.dirname(_nvcc())), "include"),
               "-o", LIB_HOST, *srcs,
               "-L", PKG, "-lrip_cuda", "-Wl,-rpath,$ORIGIN"]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if verbose or res.returncode:
            sys.stderr.write(res.stdout + res.stderr)
        if res.returncode:
            raise RuntimeError("g++ failed building librip_host.so")
    return LIB_HOST


def build_all(force: bool = False, verbose: bool = False) -> None:
    build_cuda(force, verbose)
    build_host(force, verbose)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--force", action="store_true")
    ap.add_argument("--verbose", action="store_true")
    a = ap.parse_args()
    build_all(a.force, a.verbose)
    print("built", LIB_CUDA)
