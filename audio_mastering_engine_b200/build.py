"""Build libame.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo snapshot)."""
from __future__ import annotations

import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = [os.path.join(HERE, "csrc", "ame.cu")]
DEPS = SRC + [os.path.join(HERE, "csrc", "ame_kernels.cuh"), os.path.join(HERE, "csrc", "ame_layout.h"),
              os.path.join(os.path.dirname(HERE), "include", "ame.h")]
OUT = os.path.join(HERE, "libame.so")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def needs_build() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(d) > t for d in DEPS)


def build(force: bool = False, verbose: bool = False) -> str:
    if force or needs_build():
        nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", OUT] + SRC + ["-ldl"]
        subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    import sys
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
