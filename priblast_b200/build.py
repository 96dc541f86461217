"""Builds libpriblast_acc.so in-tree with nvcc for sm_100a (no JIT cache, no torch extension machinery:
the library is a plain C-ABI shared object so non-Python hosts can link it)."""
from __future__ import annotations

import os
import shutil
import subprocess

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libpriblast_acc.so")
BLOB = os.path.join(PKG, "data", "turner99.bin")
HOST_CXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
HOST_CC = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O2",
    "-ccbin", HOST_CXX,
]

SOURCES = ["acc_kernels.cu", "acc_exact.cu", "acc_wide.cu", "sa_gpu.cu", "acc_tables.cpp"]
# the exact engine reproduces the reference's IEEE arithmetic bit for bit: no FMA contraction in that TU
PER_SOURCE_FLAGS = {"acc_exact.cu": ["-fmad=false"]}
DEPS = SOURCES + ["acc_core.h", "acc_tile.h", "acc_tables.h", "acc_exact.h", "acc_wide.h", "turner_params.h", "turner_blob.c",
                  os.path.join("..", "..", "include", "priblast_acc.h")]


def nvcc_path() -> str:
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found: libpriblast_acc.so cannot be built (there is no CPU fallback)")
    return p


def is_stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in DEPS) or os.path.getmtime(BLOB) > t


def build_library(force: bool = False, verbose: bool = False, extra: list[str] | None = None) -> str:
    if not force and not is_stale():
        return LIB
    from concurrent.futures import ThreadPoolExecutor
    blob_obj = os.path.join(CSRC, "turner_blob.o")
    subprocess.run([HOST_CC, "-O2", "-fPIC", "-c", os.path.join(CSRC, "turner_blob.c"),
                    f'-DPRIB_TURNER_BIN="{BLOB}"', "-o", blob_obj], check=True)
    nvcc = nvcc_path()

    def compile_one(src: str) -> str:  # one object per source, compiled side by side (CUB makes sa_gpu.cu slow)
        obj = os.path.join(CSRC, os.path.splitext(src)[0] + ".o")
        cmd = [nvcc, *NVCC_FLAGS, *PER_SOURCE_FLAGS.get(src, []), *(extra or []), "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            print(" ".join(cmd))
        subprocess.run(cmd, check=True)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, *NVCC_FLAGS, "-shared", *objs, blob_obj, "-o", LIB]
    if verbose:
        print(" ".join(cmd))
    subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    import sys
    print(build_library(force=True, verbose=True, extra=sys.argv[1:]))
