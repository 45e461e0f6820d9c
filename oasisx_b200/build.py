"""Build libb200ipcs.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "csrc", "b200ipcs.cu")
LIB = os.path.join(HERE, "libb200ipcs.so")
DEPS = [SRC] + [os.path.join(HERE, "csrc", f) for f in ("common.cuh", "elem.cuh", "linalg.cuh", "mg.cuh", "amg.cuh", "gmres.cuh", "ref_tables.h")] + [
    os.path.join(os.path.dirname(HERE), "include", "b200ipcs.h")
]


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(d) > t for d in DEPS if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [
        nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
        "-Xcompiler", "-fPIC", "-shared", "-o", LIB, SRC, "-lcudart",
    ]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed building libb200ipcs.so")
    if verbose:
        sys.stderr.write(res.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
