"""Builds libd2pc.so (the C-ABI CUDA library, include/d2pc.h) in-tree with nvcc for sm_100a.

nvcc cross-compiles without a GPU, so this runs in the build container; the resulting
``image_to_pointcloud_b200/_build/libd2pc.so`` is git-ignored but travels to the GPU box.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
BUILD_DIR = os.path.join(PKG_DIR, "_build")
LIB_PATH = os.path.join(BUILD_DIR, "libd2pc.so")
SOURCES = ["d2pc_api.cu", "d2pc_stats.cu", "d2pc_emit.cu", "d2pc_path.cu", "d2pc_voxel.cu", "d2pc_serialise.cu", "d2pc_sor.cu",
           "d2pc_normals.cu", "d2pc_mesh.cu", "d2pc_simplify.cu", "d2pc_components.cu",
           "d2pc_smooth.cu", "d2pc_cluster.cu"]
HEADERS = ["d2pc_math.h", "d2pc_format.h", "d2pc_device.cuh", "d2pc_stats_dev.cuh", "d2pc_emit_dev.cuh", "d2pc_grid.cuh",
           "d2pc_scan.cuh", "d2pc_components.h", "d2pc_smooth.h",
           os.path.join("..", "..", "include", "d2pc.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "--fmad=false",            # no implicit contraction: the float64 chain must round like NumPy
    "-Xcompiler", "-fPIC", "-shared",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (needed to build libd2pc.so)")


def source_digest() -> str:
    h = hashlib.sha256()
    for name in SOURCES + HEADERS:
        with open(os.path.join(CSRC, name), "rb") as f:
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def stored_digest() -> str:
    """Digest of the sources the in-tree library was built from ("" if unknown)."""
    try:
        return open(os.path.join(BUILD_DIR, "libd2pc.sha256")).read().strip()
    except OSError:
        return ""


def build_library(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(BUILD_DIR, exist_ok=True)
    stamp = os.path.join(BUILD_DIR, "libd2pc.sha256")
    digest = source_digest()
    if not force and os.path.exists(LIB_PATH) and os.path.exists(stamp):
        if open(stamp).read().strip() == digest:
            return LIB_PATH
    # one nvcc per translation unit, in parallel, then one link step
    from concurrent.futures import ThreadPoolExecutor
    nvcc = _nvcc()
    compile_flags = [f for f in NVCC_FLAGS if f != "-shared"] + (["-Xptxas", "-v"] if verbose else [])

    def compile_one(src):
        obj = os.path.join(BUILD_DIR, os.path.splitext(src)[0] + ".o")
        res = subprocess.run([nvcc] + compile_flags + ["-c", os.path.join(CSRC, src), "-o", obj],
                             capture_output=True, text=True)
        return src, obj, res

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as pool:
        results = list(pool.map(compile_one, SOURCES))
    for src, _, res in results:
        if res.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n" + res.stdout + res.stderr)
        if verbose:
            print(res.stderr)
    res = subprocess.run([nvcc, "-shared", "-Xcompiler", "-fPIC", "-gencode", "arch=compute_100a,code=sm_100a"] +
                         [obj for _, obj, _ in results] + ["-o", LIB_PATH], capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc link failed:\n" + res.stdout + res.stderr)
    with open(stamp, "w") as f:
        f.write(digest)
    return LIB_PATH


if __name__ == "__main__":
    import sys
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
