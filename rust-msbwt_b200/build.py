"""In-tree nvcc build of the engine's shared library (sm_100a only).

    python rust-msbwt_b200/build.py [--force] [--verbose]

Output: rust-msbwt_b200/libmsbwt_b200.so (git-ignored, travels to the GPU box with
the gpurun snapshot).  No torch, no JIT cache: a plain `nvcc -shared`.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libmsbwt_b200.so")
SOURCES = ["capi.cu", "hostpath.cu", "kernels.cu", "quad_kernels.cu", "stats_kernels.cu", "wide_kernels.cu", "final_kernels.cu", "ext_kernels.cu", "loader.cu", "builder.cu", "pair_builder.cu", "quad_builder.cu", "oct_builder.cu", "fin_builder.cu", "bwt_build.cu", "bwt_merge.cu", "spectrum.cu", "unitigs.cu", "correct.cu"]
HOST_SOURCES = ["hostpack.cpp", "codec.cpp"]  # plain g++ (AVX2 intrinsics behind a runtime check)
HEADERS = ["engine.h", "handle.h", "layout.h", "device_rank.cuh", "kernel_common.cuh", "pack_common.cuh", "oct_kernel.cuh", "hostpack.h", os.path.join(ROOT, "include", "msbwt_gpu.h")]

NVCC_FLAGS = [
    "-O3", "-std=c++17",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "-Xcompiler", "-fPIC,-O3,-Wall,-Wextra",
    "-shared",
]


def nvcc_path() -> str:
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found: the engine has no CPU fallback and cannot be built without it")
    return p


def is_stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HOST_SOURCES] + [h if os.path.isabs(h) else os.path.join(CSRC, h) for h in HEADERS]
    deps.append(os.path.abspath(__file__))
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    have_sources = all(os.path.exists(os.path.join(CSRC, s)) for s in SOURCES)
    if not force and not is_stale():
        return LIB
    if not have_sources:
        raise RuntimeError("engine sources missing")
    objs = []
    for src in HOST_SOURCES:
        obj = os.path.join(CSRC, os.path.splitext(src)[0] + ".o")
        res = subprocess.run(["g++", "-O3", "-std=c++17", "-fPIC", "-Wall", "-Wextra", "-pthread", "-c",
                              os.path.join(CSRC, src), "-o", obj], capture_output=True, text=True)
        if res.returncode != 0:
            sys.stderr.write(res.stdout + res.stderr)
            raise RuntimeError("g++ failed")
        objs.append(obj)
    cmd = [nvcc_path(), *NVCC_FLAGS]
    if verbose:
        cmd += ["-Xptxas", "-v"]
    cmd += ["-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES] + objs
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed")
    if verbose:
        sys.stderr.write(res.stdout + res.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
