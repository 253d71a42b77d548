"""Build librbg_b200.so (all CUDA kernels + the C-ABI) in-tree with nvcc for sm_100a.

Usage: python routing-board-generation_b200/build.py [--force]
The .so lands in routing-board-generation_b200/lib/ (git-ignored, shipped to the GPU box).
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
SO = os.path.join(LIBDIR, "librbg_b200.so")
SOURCES = ["c_api.cu", "prw_kernel.cu", "connector_kernel.cu", "misc_kernels.cu", "seedext_kernel.cu", "seqrw_kernel.cu", "host_pool.cpp"]
CXX_FLAGS = ["-O3", "-std=c++17", "-fPIC", "-pthread"]  # plain C++ sources (host threads of the transport layer): g++
HEADERS = ["rbg_device.cuh", "connector_device.cuh", "obs_stage.cuh", "gen_warp.cuh", "select.cuh", "rbg_host.h", os.path.join("..", "..", "include", "rbg_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "--fmad=false",              # float32 parity with XLA: no contraction in the choice / reward arithmetic
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O2",
    "-Xptxas", "-v",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def is_stale() -> bool:
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    extra = os.environ.get("RBG_NVCC_EXTRA", "").split()  # extra nvcc flags, passed through as given (no source file has -D switches of its own)
    if not force and not extra and not is_stale():
        return SO
    os.makedirs(LIBDIR, exist_ok=True)
    objs = []
    logs = []
    procs = []
    for s in SOURCES:
        obj = os.path.join(LIBDIR, os.path.splitext(s)[0] + ".o")
        if s.endswith(".cpp"):
            cmd = [os.environ.get("CXX", "g++"), *CXX_FLAGS, "-c", os.path.join(CSRC, s), "-o", obj]
        else:
            cmd = [_nvcc(), *NVCC_FLAGS, *extra, "-c", os.path.join(CSRC, s), "-o", obj]
        procs.append((s, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for s, obj, pr in procs:
        out, _ = pr.communicate()
        logs.append(f"==== {s}\n{out}")
        if pr.returncode != 0:
            raise RuntimeError(f"nvcc failed on {s}:\n{out}")
        objs.append(obj)
    link = [_nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", SO, *objs, "-lcudart_static", "-lpthread", "-ldl", "-lrt"]
    r = subprocess.run(link, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}{r.stderr}")
    with open(os.path.join(LIBDIR, "build.log"), "w") as f:
        f.write("\n".join(logs))
    if verbose:
        print("\n".join(logs))
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
