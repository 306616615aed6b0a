"""Builds and binds tests/hostsmooth/hostsmooth.cpp (the product's d2pc_smooth.h compiled for the host).  The library
goes to a temporary directory: the tests must not write into the tree."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import d2pc_smooth_oracle as SMO

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "hostsmooth.cpp")
CSRC = os.path.join(HERE, "..", "..", "image_to_pointcloud_b200", "csrc")
HDRS = [os.path.join(CSRC, n) for n in ("d2pc_smooth.h", "d2pc_math.h")] + \
    [os.path.join(HERE, "..", "..", "include", "d2pc.h")]
FLAGS = ["-O2", "-ffp-contract=off", "-fPIC", "-shared", "-std=c++17"]
FIELD_BITS = {"vertex": 1, "normal": 2, "color": 4}

_lib = None


def build():
    h = hashlib.sha256(" ".join(FLAGS).encode())
    for p in [SRC] + HDRS:
        with open(p, "rb") as f:
            h.update(f.read())
    so = os.path.join(tempfile.gettempdir(), f"d2pc_hostsmooth_{os.getuid()}_{h.hexdigest()[:16]}.so")
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
        lib.hs_smooth.restype = None
        lib.hs_smooth.argtypes = [vp, vp, vp, C.c_uint32, vp, vp, C.c_int, vp, C.c_uint32, C.c_uint32, vp, vp, vp]
        lib.hs_normals.restype = None
        lib.hs_normals.argtypes = [vp, C.c_uint32, vp, C.c_uint32, vp, vp, vp]
        _lib = lib
    return _lib


def smooth(mesh, method, iterations=1, lambda_filter=0.5, mu=-0.53, scope="all"):
    """The oracle's Mesh layout, computed by d2pc_smooth.h over the oracle's adjacency."""
    lib = load()
    v = np.ascontiguousarray(mesh.vertices, np.float32).reshape(-1, 3)
    c = np.ascontiguousarray(mesh.colors, np.float32).reshape(-1, 3)
    n = None if mesh.vertex_normals is None else np.ascontiguousarray(mesh.vertex_normals, np.float64).reshape(-1, 3)
    t = np.ascontiguousarray(mesh.triangles, np.int32).reshape(-1, 3)
    V = len(v)
    off, nbr = SMO.adjacency(V, t)
    off, nbr = np.ascontiguousarray(off, np.uint32), np.ascontiguousarray(nbr, np.uint32)
    lams = [lam for _, lam in SMO._passes(method, iterations, lambda_filter, mu)]
    lams = np.ascontiguousarray(lams if lams else [0.0], np.float64)
    fields = sum(FIELD_BITS[f] for f in SMO.SCOPES[scope] if f != "normal" or n is not None)
    passes = len(lams) if SMO._passes(method, iterations, lambda_filter, mu) else 0
    ov, oc = v.copy(), c.copy()
    on = None if n is None else n.copy()
    if passes and fields and V:
        lib.hs_smooth(v.ctypes.data, c.ctypes.data, None if n is None else n.ctypes.data, V, off.ctypes.data,
                      nbr.ctypes.data, int(method != "simple"), lams.ctypes.data, passes, fields, ov.ctypes.data,
                      oc.ctypes.data, None if on is None else on.ctypes.data)
    return SMO.Mesh(ov, oc, t, on, np.asarray(mesh.vertex_rows, np.int64).reshape(-1))


def normals(mesh):
    """compute_vertex_normals through d2pc_smooth.h over a (vertex, triangle) incidence in ascending triangle order."""
    lib = load()
    v = np.ascontiguousarray(mesh.vertices, np.float32).reshape(-1, 3)
    t = np.ascontiguousarray(mesh.triangles, np.int32).reshape(-1, 3)
    V, T = len(v), len(t)
    vids = t.reshape(-1).astype(np.int64)
    order = np.argsort(vids, kind="stable")
    tri = np.ascontiguousarray(order // 3, np.uint32)
    off = np.zeros(V + 1, np.uint32)
    np.cumsum(np.bincount(vids, minlength=V), out=off[1:])
    out = np.zeros((V, 3), np.float64)
    if V:
        lib.hs_normals(v.ctypes.data, V, t.ctypes.data, T, off.ctypes.data, tri.ctypes.data, out.ctypes.data)
    return out
