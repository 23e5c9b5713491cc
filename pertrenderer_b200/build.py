"""Build the sm_100a shared library of the perturbed shading kernels, in-tree.

    python -m pertrenderer_b200.build [--force]

Produces ``pertrenderer_b200/libpertshade.so`` (git-ignored, travels to the GPU box with the
repository snapshot).  nvcc cross-compiles without a GPU.
"""

from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC_DIR = os.path.join(HERE, "csrc")
SOURCES = [os.path.join(SRC_DIR, f) for f in ("cabi.cu", "shade_fwd.cu", "shade_bwd.cu", "shade_soft.cu", "ops_standalone.cu", "phong.cu", "raster.cu")]
HEADERS = [os.path.join(SRC_DIR, f) for f in ("philox.cuh", "common.cuh", "tile.cuh", "texel.cuh", "kernels.h")] + \
    [os.path.join(os.path.dirname(HERE), "include", "pertshade.h")]
LIB_PATH = os.path.join(HERE, "libpertshade.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
    # no --use_fast_math: the explicit-noise parity mode needs IEEE division / logf and
    # uncontracted multiply-add where the kernels ask for it (__fmul_rn / __fadd_rn)
]


def find_nvcc() -> str:
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: cannot build libpertshade.so")
    return nvcc


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(p) > t for p in SOURCES + HEADERS)


def build_library(force: bool = False, verbose: bool = False) -> str:
    """Compile every translation unit (in parallel) and link libpertshade.so in-tree."""
    if not force and not is_stale():
        return LIB_PATH
    import concurrent.futures
    nvcc = find_nvcc()
    obj_dir = os.path.join(os.path.dirname(HERE), "build")
    os.makedirs(obj_dir, exist_ok=True)
    compile_flags = [f for f in NVCC_FLAGS if f != "-shared"]

    def compile_one(src):
        obj = os.path.join(obj_dir, os.path.basename(src)[:-3] + ".o")
        cmd = [nvcc] + compile_flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, src]
        proc = subprocess.run(cmd, capture_output=True, text=True)
        if proc.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + proc.stdout + proc.stderr)
        return obj, proc.stderr

    with concurrent.futures.ThreadPoolExecutor(max_workers=len(SOURCES)) as pool:
        results = list(pool.map(compile_one, SOURCES))
    if verbose:
        for _, err in results:
            print(err)
    cmd = [nvcc, "-shared", "-Xcompiler", "-fPIC", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB_PATH] + \
        [o for o, _ in results]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError("link failed:\n" + " ".join(cmd) + "\n" + proc.stdout + proc.stderr)
    return LIB_PATH


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
