"""Builds liblmc_b200.so (hand-written sm_100a CUDA + C ABI) in-tree with nvcc.

nvcc cross-compiles without a GPU; the .so is git-ignored but travels with the tree."""
from __future__ import annotations

import glob
import os
import shutil
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.environ.get("LMC_B200_LIB_OUT") or os.path.join(PKG_DIR, "liblmc_b200.so")   # (_LIB_OUT: experiment builds)

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC",
]
OBJ_DIR = os.environ.get("LMC_B200_OBJ_DIR") or os.path.join(PKG_DIR, "build")          # git-ignored


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = sources() + glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(CSRC, "*.h")) + [os.path.join(PKG_DIR, "..", "include", "lmc_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB_PATH
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: liblmc_b200.so cannot be built (there is no CPU fallback)")
    # one nvcc per translation unit, in parallel (the streaming kernels dominate: ~40 s), then one link
    from concurrent.futures import ThreadPoolExecutor
    os.makedirs(OBJ_DIR, exist_ok=True)
    extra = (["-Xptxas", "-v"] if verbose else []) + [f for f in os.environ.get("LMC_NVCC_EXTRA", "").split() if f]

    def compile_one(src):
        obj = os.path.join(OBJ_DIR, os.path.basename(src)[:-3] + ".o")
        r = subprocess.run([nvcc] + NVCC_FLAGS + extra + ["-c", src, "-o", obj], capture_output=True, text=True)
        return src, obj, r
    with ThreadPoolExecutor(max(1, min(len(sources()), os.cpu_count() or 1))) as ex:
        results = list(ex.map(compile_one, sources()))
    for src, _, r in results:
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n" + r.stdout + r.stderr)
        if verbose:
            print(r.stderr)
    tmp = LIB_PATH + ".tmp"
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", tmp] + [o for _, o, _ in results],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    os.replace(tmp, LIB_PATH)
    return LIB_PATH


if __name__ == "__main__":
    print(build_library(force=True, verbose=True))
