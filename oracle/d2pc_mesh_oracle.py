"""TEST INFRASTRUCTURE ONLY -- CPU oracle for the lattice mesh (DESIGN row m1): a triangle mesh of one frame's
unmasked emit rows, using the image lattice the rows come from, and its Open3D-layout mesh PLY.

SPEC FROZEN HERE, NO REFERENCE CODE: the reference builds meshes with normals + Poisson / BPA (backend/app.py:271-308,
508-535); this is our own depth-image triangulation, with the same status as the depth-range mask (ax-1) and the voxel
grid (ax-2).  Its vertex normals and PLY layout restate Open3D's published source (geometry/TriangleMesh.cpp
``ComputeVertexNormals(normalized=True)``, io/file_format/FilePLY.cpp ``WriteTriangleMeshToPLY``); Open3D is not
installed in the build container, so that part is PARITY UNPINNED, as in ``d2pc_normals_oracle``.  The product
package never imports it.

Spec (row i = r * C + c of an R x C lattice):
  valid      keep[i] (when given) and all three coordinates finite
  quads      q = r * (C - 1) + c with corners a = (r, c), b = (r, c + 1), p = (r + 1, c), d = (r + 1, c + 1)
             4 valid corners: d2(a, d) <= d2(b, p) -> T0 = (a, p, d), T1 = (a, d, b); else T0 = (a, p, b), T1 = (b, p, d)
             3 valid corners: one candidate, d missing (a, p, b), a missing (b, p, d), b missing (a, p, d),
             p missing (a, d, b); fewer: none
  filter     float64, in this order: n = (p1 - p0) x (p2 - p0) (Eigen's component order), n.n > 0;
             s = (p0 + p1) + p2, n.s < 0; (n.s)^2 >= cos2 * (n.n) * (s.s); with max_edge every edge's d2 <= max_edge^2
  order      triangles by quad, T0 before T1; vertices the valid rows (referenced by a kept triangle with
             remove_unreferenced) in lattice order; triangles as int32 vertex ids
  normals    sum of the unnormalised n of the adjacent kept triangles in ascending triangle order, from zero;
             v / sqrt(v.v), (0, 0, 1) for a zero sum
"""
from __future__ import annotations

import math
from typing import NamedTuple, Optional

import numpy as np

from .d2pc_normals_oracle import PLY_NORMAL_HEADER, _axiswise_d2, ply_normal_records
from .d2pc_oracle import F64, PLY_HEADER, ply_records


class Mesh(NamedTuple):
    vertices: np.ndarray         # float32 [V, 3]
    colors: np.ndarray           # float32 [V, 3]
    triangles: np.ndarray        # int32 [T, 3]
    vertex_normals: Optional[np.ndarray]   # float64 [V, 3] or None
    vertex_rows: np.ndarray      # int64 [V]


# corners a, b, p, d = 0, 1, 2, 3; the candidate triangles of every quad configuration (None: no T1)
QUAD_TRIANGLES = {
    "ad": ((0, 2, 3), (0, 3, 1)),
    "bp": ((0, 2, 1), (1, 2, 3)),
    "no_d": ((0, 2, 1), None),
    "no_a": ((1, 2, 3), None),
    "no_b": ((0, 2, 3), None),
    "no_p": ((0, 3, 1), None),
}


def cos2_of(max_angle: float) -> float:
    """cos(radians(max_angle))^2 as the host computes it once (Python floats)."""
    c = math.cos(math.radians(float(max_angle)))
    return c * c


def valid_rows(xyz: np.ndarray, keep: Optional[np.ndarray] = None) -> np.ndarray:
    ok = np.isfinite(np.asarray(xyz, dtype=np.float32)).all(axis=1)
    if keep is not None:
        ok &= np.asarray(keep).reshape(-1).astype(bool)
    return ok


def _cross(a, b):
    return np.stack([a[:, 1] * b[:, 2] - a[:, 2] * b[:, 1], a[:, 2] * b[:, 0] - a[:, 0] * b[:, 2],
                     a[:, 0] * b[:, 1] - a[:, 1] * b[:, 0]], axis=1)


def _dot(a, b):
    return a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1] + a[:, 2] * b[:, 2]


def triangle_normals(p0: np.ndarray, p1: np.ndarray, p2: np.ndarray) -> np.ndarray:
    """Unnormalised n = (p1 - p0) x (p2 - p0) in float64 (Open3D ``ComputeTriangleNormals(false)``)."""
    return _cross(p1 - p0, p2 - p0)


def triangle_keep(p0, p1, p2, cos2: float, max_edge2: Optional[float]) -> np.ndarray:
    """The filter on float64 corners [m, 3]."""
    n = triangle_normals(p0, p1, p2)
    nn = _dot(n, n)
    s = (p0 + p1) + p2
    ns = _dot(n, s)
    ss = _dot(s, s)
    ok = (nn > 0.0) & (ns < 0.0) & (ns * ns >= cos2 * nn * ss)
    if max_edge2 is not None:
        ok &= (_axiswise_d2(p0, p1) <= max_edge2) & (_axiswise_d2(p1, p2) <= max_edge2) & \
              (_axiswise_d2(p2, p0) <= max_edge2)
    return ok


def _edge2(max_edge) -> Optional[float]:
    return None if max_edge is None else float(max_edge) * float(max_edge)


def _finish(xyz, rgb, n_rows, valid, tri_rows, remove_unreferenced, compute_normals):
    """Kept triangles as lattice rows [T, 3] (in order) -> Mesh."""
    if remove_unreferenced:
        vert = np.zeros(n_rows, bool)
        vert[tri_rows.reshape(-1)] = True
    else:
        vert = valid
    rows = np.nonzero(vert)[0].astype(np.int64)
    idmap = np.full(n_rows, -1, np.int64)
    idmap[rows] = np.arange(len(rows))
    tris = idmap[tri_rows].astype(np.int32).reshape(-1, 3)
    normals = None
    if compute_normals:
        p = np.asarray(xyz, np.float32).astype(F64)
        tn = triangle_normals(p[tri_rows[:, 0]], p[tri_rows[:, 1]], p[tri_rows[:, 2]]) if len(tri_rows) else \
            np.zeros((0, 3))
        vids = tris.reshape(-1).astype(np.int64)
        contrib = np.repeat(tn, 3, axis=0)
        order = np.argsort(vids, kind="stable")          # per vertex: ascending triangle order
        vs, cs = vids[order], contrib[order]
        first = np.searchsorted(vs, vs, side="left")
        rank = np.arange(len(vs)) - first
        acc = np.zeros((len(rows), 3))
        for k in range(int(rank.max()) + 1 if len(rank) else 0):
            sel = rank == k
            acc[vs[sel]] = acc[vs[sel]] + cs[sel]
        normals = normalise(acc)
    return Mesh(np.asarray(xyz, np.float32)[rows], np.asarray(rgb, np.float32)[rows], tris, normals, rows)


def normalise(acc: np.ndarray) -> np.ndarray:
    s = _dot(acc, acc)
    with np.errstate(all="ignore"):
        out = acc / np.sqrt(s)[:, None]
    out[s == 0.0] = [0.0, 0.0, 1.0]
    return out


def grid_mesh(xyz: np.ndarray, rgb: np.ndarray, lattice_shape, keep: Optional[np.ndarray] = None,
              max_edge: Optional[float] = None, max_angle: float = 85.0, remove_unreferenced: bool = True,
              compute_normals: bool = True) -> Mesh:
    """Vectorised restatement of the spec (module docstring)."""
    R, C = int(lattice_shape[0]), int(lattice_shape[1])
    xyz = np.asarray(xyz, np.float32).reshape(-1, 3)
    assert len(xyz) == R * C
    valid = valid_rows(xyz, keep)
    p = xyz.astype(F64)
    cos2, me2 = cos2_of(max_angle), _edge2(max_edge)
    if R >= 2 and C >= 2:
        r, c = np.mgrid[0:R - 1, 0:C - 1]
        ia = (r * C + c).reshape(-1).astype(np.int64)
        corner = np.stack([ia, ia + 1, ia + C, ia + C + 1], axis=1)      # a, b, p, d
        v = valid[corner]
        nv = v.sum(axis=1)
        with np.errstate(invalid="ignore"):                              # invalid corners: NaN, never used
            ad = _axiswise_d2(p[corner[:, 0]], p[corner[:, 3]]) <= _axiswise_d2(p[corner[:, 1]], p[corner[:, 2]])
        Q = len(ia)
        cand = np.zeros((Q, 2, 3), np.int64)
        has = np.zeros((Q, 2), bool)
        cases = [("ad", (nv == 4) & ad), ("bp", (nv == 4) & ~ad), ("no_d", (nv == 3) & ~v[:, 3]),
                 ("no_a", (nv == 3) & ~v[:, 0]), ("no_b", (nv == 3) & ~v[:, 1]), ("no_p", (nv == 3) & ~v[:, 2])]
        for name, m in cases:
            for t, tri in enumerate(QUAD_TRIANGLES[name]):
                if tri is not None:
                    cand[m, t] = corner[m][:, list(tri)]
                    has[m, t] = True
        flat = cand.reshape(-1, 3)
        ok = has.reshape(-1).copy()
        idx = np.nonzero(ok)[0]
        ok[idx] = triangle_keep(p[flat[idx, 0]], p[flat[idx, 1]], p[flat[idx, 2]], cos2, me2)
        tri_rows = flat[ok]
    else:
        tri_rows = np.zeros((0, 3), np.int64)
    return _finish(xyz, rgb, R * C, valid, tri_rows, remove_unreferenced, compute_normals)


def grid_mesh_loop(xyz: np.ndarray, rgb: np.ndarray, lattice_shape, keep: Optional[np.ndarray] = None,
                   max_edge: Optional[float] = None, max_angle: float = 85.0, remove_unreferenced: bool = True,
                   compute_normals: bool = True) -> Mesh:
    """Plain per-quad loop over Python floats: the second restatement the vectorised one is checked against."""
    R, C = int(lattice_shape[0]), int(lattice_shape[1])
    xyz = np.asarray(xyz, np.float32).reshape(-1, 3)
    valid = [bool(x) for x in valid_rows(xyz, keep)]
    P = [tuple(float(v) for v in row) for row in xyz]
    cos2 = cos2_of(max_angle)
    me2 = _edge2(max_edge)

    def d2(q, w):
        dx, dy, dz = q[0] - w[0], q[1] - w[1], q[2] - w[2]
        s = dx * dx
        s += dy * dy
        s += dz * dz
        return s

    def normal(p0, p1, p2):
        a = (p1[0] - p0[0], p1[1] - p0[1], p1[2] - p0[2])
        b = (p2[0] - p0[0], p2[1] - p0[1], p2[2] - p0[2])
        return (a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0])

    def dot(u, w):
        return u[0] * w[0] + u[1] * w[1] + u[2] * w[2]

    def keep_tri(i0, i1, i2):
        p0, p1, p2 = P[i0], P[i1], P[i2]
        n = normal(p0, p1, p2)
        nn = dot(n, n)
        if not nn > 0.0:
            return False
        s = ((p0[0] + p1[0]) + p2[0], (p0[1] + p1[1]) + p2[1], (p0[2] + p1[2]) + p2[2])
        ns = dot(n, s)
        if not ns < 0.0:
            return False
        if not ns * ns >= cos2 * nn * dot(s, s):
            return False
        if me2 is not None:
            return d2(p0, p1) <= me2 and d2(p1, p2) <= me2 and d2(p2, p0) <= me2
        return True

    tri_rows = []
    for r in range(R - 1):
        for c in range(C - 1):
            k = (r * C + c, r * C + c + 1, (r + 1) * C + c, (r + 1) * C + c + 1)
            vv = [valid[i] for i in k]
            if sum(vv) == 4:
                name = "ad" if d2(P[k[0]], P[k[3]]) <= d2(P[k[1]], P[k[2]]) else "bp"
            elif sum(vv) == 3:
                name = ("no_a", "no_b", "no_p", "no_d")[vv.index(False)]
            else:
                continue
            for tri in QUAD_TRIANGLES[name]:
                if tri is not None and keep_tri(k[tri[0]], k[tri[1]], k[tri[2]]):
                    tri_rows.append([k[tri[0]], k[tri[1]], k[tri[2]]])
    tri_rows = np.array(tri_rows, np.int64).reshape(-1, 3)
    used = set(int(i) for i in tri_rows.reshape(-1))
    rows = [i for i in range(R * C) if valid[i] and (not remove_unreferenced or i in used)]
    ids = {row: v for v, row in enumerate(rows)}
    tris = np.array([[ids[i] for i in t] for t in tri_rows], np.int32).reshape(-1, 3)
    normals = None
    if compute_normals:
        acc = [[0.0, 0.0, 0.0] for _ in rows]
        for t in tri_rows:
            n = normal(P[t[0]], P[t[1]], P[t[2]])
            for i in t:
                a = acc[ids[int(i)]]
                a[0] += n[0]
                a[1] += n[1]
                a[2] += n[2]
        out = []
        for a in acc:
            s = dot(a, a)
            out.append([0.0, 0.0, 1.0] if s == 0.0 else [a[0] / math.sqrt(s), a[1] / math.sqrt(s), a[2] / math.sqrt(s)])
        normals = np.array(out, F64).reshape(-1, 3)
    rows = np.array(rows, np.int64)
    return Mesh(xyz[rows], np.asarray(rgb, np.float32)[rows], tris, normals, rows)


# --------------------------------------------------------------------------------------------
# mesh PLY (Open3D write_triangle_mesh, binary little endian)
# --------------------------------------------------------------------------------------------
PLY_FACE_RECORD_DTYPE = np.dtype([("n", "u1"), ("v0", "<u4"), ("v1", "<u4"), ("v2", "<u4")])
PLY_FACE_ELEMENT = "element face {m}\nproperty list uchar uint vertex_indices\n"
PLY_MESH_HEADER = PLY_HEADER.replace("end_header\n", PLY_FACE_ELEMENT + "end_header\n")
PLY_MESH_NORMAL_HEADER = PLY_NORMAL_HEADER.replace("end_header\n", PLY_FACE_ELEMENT + "end_header\n")


def ply_face_records(triangles: np.ndarray) -> np.ndarray:
    """13-byte faces: uchar 3, then the three vertex ids as uint32."""
    assert PLY_FACE_RECORD_DTYPE.itemsize == 13
    t = np.asarray(triangles).reshape(-1, 3)
    rec = np.zeros(len(t), PLY_FACE_RECORD_DTYPE)
    rec["n"] = 3
    rec["v0"], rec["v1"], rec["v2"] = t[:, 0], t[:, 1], t[:, 2]
    return rec


def mesh_ply_bytes(mesh: Mesh) -> bytes:
    """The bytes of Open3D's ``write_triangle_mesh(..., write_ascii=False)`` for the mesh: vertices (with nx, ny, nz
    after z when it has normals) and faces.  PARITY UNPINNED."""
    nv, nt = len(mesh.vertices), len(mesh.triangles)
    if mesh.vertex_normals is None:
        head = PLY_MESH_HEADER.format(n=nv, m=nt)
        vrec = ply_records(mesh.vertices, mesh.colors)
    else:
        head = PLY_MESH_NORMAL_HEADER.format(n=nv, m=nt)
        vrec = ply_normal_records(mesh.vertices, mesh.vertex_normals, mesh.colors)
    return head.encode("ascii") + vrec.tobytes() + ply_face_records(mesh.triangles).tobytes()
