"""Builds and binds tests/hostcomp/hostcomp.cpp (the product's d2pc_components.h compiled for the host).  The
library goes to a temporary directory: the tests must not write into the tree."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "hostcomp.cpp")
CSRC = os.path.join(HERE, "..", "..", "image_to_pointcloud_b200", "csrc")
HDRS = [os.path.join(CSRC, n) for n in ("d2pc_components.h", "d2pc_math.h")] + \
    [os.path.join(HERE, "..", "..", "include", "d2pc.h")]
FLAGS = ["-O2", "-ffp-contract=off", "-fPIC", "-shared", "-std=c++17"]

_lib = None


def build():
    h = hashlib.sha256(" ".join(FLAGS).encode())
    for p in [SRC] + HDRS:
        with open(p, "rb") as f:
            h.update(f.read())
    so = os.path.join(tempfile.gettempdir(), f"d2pc_hostcomp_{os.getuid()}_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.run(["g++"] + FLAGS + [SRC, "-o", tmp], check=True)
        os.replace(tmp, so)
    return so


def load():
    global _lib
    if _lib is None:
        lib = C.CDLL(build())
        vp = C.c_void_p
        lib.hc_components.restype = C.c_long
        lib.hc_components.argtypes = [vp, C.c_uint32, vp, C.c_uint32, C.c_uint64, vp, vp, vp, vp, vp]
        lib.hc_insert_full.argtypes = [C.c_uint32]
        lib.hc_chain_bounds.argtypes = [C.c_uint32]
        _lib = lib
    return _lib


def components(mesh, seed):
    """(labels int32 [T], n int64 [K], area float64 [K], error word) through the shared header."""
    lib = load()
    v = np.ascontiguousarray(mesh.vertices, np.float32).reshape(-1, 3)
    t = np.ascontiguousarray(mesh.triangles, np.int32).reshape(-1, 3)
    T = len(t)
    lab = np.zeros(max(T, 1), np.int32)
    n = np.zeros(max(T, 1), np.int64)
    area = np.zeros(max(T, 1), np.float64)
    k, err = C.c_uint32(0), C.c_int32(0)
    lib.hc_components(v.ctypes.data, len(v), t.ctypes.data, T, seed, lab.ctypes.data, n.ctypes.data,
                      area.ctypes.data, C.byref(k), C.byref(err))
    K = int(k.value)
    return lab[:T], n[:K], area[:K], int(err.value)
