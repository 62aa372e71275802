"""Build ml2048_b200/libml2048_b200.so for sm_100a with nvcc (in-tree, so it travels to the GPU box)."""

from __future__ import annotations

import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(_HERE, "csrc", "vecgame_kernels.cu")
HOST_SRC = os.path.join(_HERE, "csrc", "host_pcg64.cpp")
HOST_UNPACK_SRC = os.path.join(_HERE, "csrc", "host_unpack.cpp")
COMPRESSIBLE_SRC = os.path.join(_HERE, "csrc", "compressible_alloc.cpp")
DEPS = [SRC, HOST_SRC, HOST_UNPACK_SRC, COMPRESSIBLE_SRC, os.path.join(_HERE, "csrc", "board_ops.cuh"), os.path.join(os.path.dirname(_HERE), "include", "ml2048_b200.h")]
LIB = os.path.join(_HERE, "libml2048_b200.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-shared", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
    "-cudart", "static",
]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA extension cannot be built")


def up_to_date() -> bool:
    return os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(d) for d in DEPS)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and up_to_date() and not os.environ.get("ML2048_NVCC_EXTRA"):
        return LIB
    extra = os.environ.get("ML2048_NVCC_EXTRA", "").split()  # experiment switches, e.g. -DML2048_STORE_DEFAULT
    cmd = [nvcc_path(), *NVCC_FLAGS, *extra, "-o", LIB, SRC, HOST_SRC, HOST_UNPACK_SRC, COMPRESSIBLE_SRC]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    import sys

    print(build(force=True, verbose="-v" in sys.argv))
