"""In-tree build of the CUDA shared library (nvcc, sm_100a only)."""
from __future__ import annotations

import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.path.join(HERE, "libinversus_b200.so")
SOURCES = [os.path.join(CSRC, "inversus_b200.cu"), os.path.join(CSRC, "policy_kernels.cu"),
           os.path.join(CSRC, "encoder_kernels.cu"), os.path.join(CSRC, "wgrad_kernels.cu"),
           os.path.join(CSRC, "eval_kernels.cu")]
HOST_SOURCES = [os.path.join(CSRC, "host_expand.cpp")]  # plain C++ (AVX2 intrinsics), compiled by g++
DEPS = SOURCES + HOST_SOURCES + [os.path.join(CSRC, "inversus_kernels.cuh"), os.path.join(CSRC, "launch_common.h"),
                  os.path.join(os.path.dirname(HERE), "include", "inversus_b200.h")]

# --cudart=shared: the artefact links libcudart dynamically instead of embedding the whole runtime
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "-shared", "--cudart=shared"]


def find_nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: cannot build libinversus_b200.so")


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(d) > t for d in DEPS)


def build_library(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/*.cu into libinversus_b200.so next to this file. Cross-compiles without a GPU."""
    if force or is_stale():
        objs = []
        for src in HOST_SOURCES:
            obj = os.path.join(HERE, os.path.basename(src) + ".o")
            cmd = ["g++", "-O3", "-std=c++17", "-fPIC", "-pthread", "-c", src, "-o", obj]
            if verbose:
                print(" ".join(cmd))
            subprocess.check_call(cmd)
            objs.append(obj)
        cmd = [find_nvcc()] + NVCC_FLAGS + ["-o", LIB_PATH] + SOURCES + objs
        if verbose:
            print(" ".join(cmd))
        subprocess.check_call(cmd)
    return LIB_PATH
