"""TEST INFRASTRUCTURE ONLY -- CPU oracle for mesh simplification by vertex clustering (DESIGN row m2).

SPEC FROZEN HERE, NO REFERENCE CODE: the reference simplifies its Poisson mesh for the browser preview with Open3D
(backend/app.py:271-308, 508-535).  This is our own data-parallel rule, modelled on Open3D's
``TriangleMesh::SimplifyVertexClustering`` (geometry/TriangleMeshSimplification.cpp) and Lindstrom's out-of-core
quadric placement; Open3D is not installed in the build container, so parity is UNPINNED.  The product package
never imports this module.

Input: a mesh in the ``TriangleMesh`` layout (vertices f32 [V, 3], colors f32 [V, 3], triangles i32 [T, 3],
vertex_normals f64 [V, 3] or None, vertex_rows i64 [V]), a voxel size ``vs`` (finite, > 0) and a contraction,
"average" or "quadric".

  errors      a vertex with a non-finite coordinate, colour or normal; a triangle id outside [0, V); a cluster
              index >= 2^21 (ValueError)
  index       bmin = per-axis minimum of the float64 vertices, vmin = bmin - vs/2, idx = floor((v - vmin) / vs): the
              ax-2 voxel rule (``d2pc_oracle.voxel_indices``)
  vertices    one per occupied cluster, ordered by the lowest member vertex id; its vertex_rows entry is that
              member's (Open3D leaves the order to an unordered_map)
  colours,    exact sum / count, rounded to float64, then to float32
  average
  normals     exact sum of the members' normals rounded to float64, divided by its float64 norm (Eigen's
              ``normalized()``: sqrt of x*x + y*y + z*z in that order); a zero sum stays (0, 0, 0)
  quadric     in coordinates q = float64(v) - bmin, per input triangle: c = (q1 - q0) x (q2 - q0) (Eigen's order),
              cc = c.c; skipped when cc == 0; l = sqrt(cc), w = l / 2 (the area), n = c / l, d = -(n.q0);
              A_ij += (w n_i) n_j and b_i += (w d) n_i are added to the cluster of each of its three corners, once per
              corner (a triangle with two corners in one cluster adds twice, as Open3D sums per-vertex quadrics),
              as float64 sums in (triangle, corner) order.  With t = trace(A) and det(A) from the cofactors of row 0:
              when t > 0 and det > 1e-4 t^3 the vertex is x = -adj(A) b / det + bmin, provided x lies in the
              cluster's own cell [vmin + idx vs, vmin + (idx + 1) vs] on every axis; otherwise the average.
              Departures from Open3D: it tests |det A| > 1e-4 absolutely, which at the scale of this project almost
              never passes (a cluster of area a has det <= (a/3)^3: 4e-8 for a 0.1-unit patch), so the same
              threshold is applied to A / trace(A); and it has no containment test, without which a near-singular
              cluster throws its vertex far away.
  triangles   corners mapped to cluster ids; dropped when two ids are equal; canonical form = the rotation that
              starts at the smallest id (orientation kept); only the first triangle of each canonical form, by input
              index, stays; output in input order, in canonical form (as Open3D writes them).  Reversed-orientation
              twins both stay, and clusters no triangle uses stay (both as in Open3D).

Two restatements: ``simplify_mesh`` (vectorised) and ``simplify_mesh_loop`` (per cluster / per triangle, exact
rational sums), which the CPU tests check against each other.
"""
from __future__ import annotations

import math
from fractions import Fraction
from typing import Optional

import numpy as np

from .d2pc_mesh_oracle import Mesh
from .d2pc_oracle import F64, VOXEL_INDEX_BITS

CONTRACTIONS = ("average", "quadric")
DET_REL = 1e-4


def _check(mesh, vs: float, contraction: str):
    vs = float(vs)
    if not (math.isfinite(vs) and vs > 0.0):
        raise ValueError("voxel_size must be a positive finite number")
    if contraction not in CONTRACTIONS:
        raise ValueError(f"contraction must be one of {CONTRACTIONS}")
    v = np.asarray(mesh.vertices, np.float32).reshape(-1, 3)
    c = np.asarray(mesh.colors, np.float32).reshape(-1, 3)
    t = np.asarray(mesh.triangles).reshape(-1, 3).astype(np.int64)
    nrm = None if mesh.vertex_normals is None else np.asarray(mesh.vertex_normals, F64).reshape(-1, 3)
    rows = np.asarray(mesh.vertex_rows, np.int64).reshape(-1)
    ok = np.isfinite(v).all() and np.isfinite(c).all() and (nrm is None or np.isfinite(nrm).all())
    if not ok:
        raise ValueError("the mesh has a non-finite vertex")
    if len(t) and (t.min() < 0 or t.max() >= len(v)):
        raise ValueError("a triangle refers to a vertex that does not exist")
    return vs, v, c, t, nrm, rows


def cluster_index(v: np.ndarray, vs: float):
    """-> (idx int64 [V, 3], bmin f64 [3], vmin f64 [3]); ValueError past 2^21 - 1."""
    p = v.astype(F64)
    bmin = p.min(axis=0)
    vmin = bmin - vs * 0.5
    idx = np.floor((p - vmin[None, :]) / vs).astype(np.int64)
    if idx.size and idx.max() >= (1 << VOXEL_INDEX_BITS):
        raise ValueError("voxel_size is too small.")
    return idx, bmin, vmin


def _clusters(idx: np.ndarray):
    """-> (cluster id of every vertex, representative (lowest) vertex of every cluster)."""
    key = (idx[:, 0] << (2 * VOXEL_INDEX_BITS)) | (idx[:, 1] << VOXEL_INDEX_BITS) | idx[:, 2]
    _, first, inv = np.unique(key, return_index=True, return_inverse=True)
    order = np.argsort(first, kind="stable")
    rank = np.empty(len(first), np.int64)
    rank[order] = np.arange(len(first))
    return rank[inv.reshape(-1)], first[order]


def _exact_sums(vals: np.ndarray, cid: np.ndarray, k: int, bits: int, mean: bool):
    """Per-cluster exact sums (mean=False: rounded to float64) or exact means (rounded to float64) of float64 columns
    that carry at most ``bits`` significant bits.  Float64 accumulation is used where it provably cannot round
    (every partial sum is a multiple of the smallest member's ulp and below 2^53 of it); the other clusters are
    summed as rationals."""
    o = np.argsort(cid, kind="stable")
    cs, vs = cid[o], vals[o]
    starts = np.searchsorted(cs, np.arange(k))
    cnt = np.diff(np.append(starts, len(cs)))
    out = np.zeros((k, vals.shape[1]))
    for j in range(vals.shape[1]):
        x = vs[:, j]
        s = np.add.reduceat(x, starts) if len(x) else np.zeros(0)
        _, e = np.frexp(x)
        nz = x != 0.0
        emax = np.maximum.reduceat(np.where(nz, e, -100000), starts) if len(x) else np.zeros(0, int)
        emin = np.minimum.reduceat(np.where(nz, e, 100000), starts) if len(x) else np.zeros(0, int)
        lg = np.ceil(np.log2(np.maximum(cnt, 1))).astype(np.int64)
        safe = (emax == -100000) | (lg + emax - (emin - bits) <= 53)
        with np.errstate(all="ignore"):
            col = s / cnt if mean else s.copy()
        for c in np.nonzero(~safe)[0]:
            seg = x[starts[c]:starts[c] + cnt[c]]
            tot = sum((Fraction(float(a)) for a in seg), Fraction(0))
            col[c] = float(tot / int(cnt[c])) if mean else float(tot)
        out[:, j] = col
    return out


def _normalise(s: np.ndarray) -> np.ndarray:
    nn = s[:, 0] * s[:, 0] + s[:, 1] * s[:, 1] + s[:, 2] * s[:, 2]
    ln = np.sqrt(nn)
    with np.errstate(all="ignore"):
        out = s / ln[:, None]
    out[nn == 0.0] = 0.0
    return out


def triangle_quadrics(q: np.ndarray, t: np.ndarray):
    """Per triangle: (A [T, 6] = a00 a01 a02 a11 a12 a22, b [T, 3], used [T]) in translated coordinates q."""
    q0, q1, q2 = q[t[:, 0]], q[t[:, 1]], q[t[:, 2]]
    e1, e2 = q1 - q0, q2 - q0
    c = np.stack([e1[:, 1] * e2[:, 2] - e1[:, 2] * e2[:, 1], e1[:, 2] * e2[:, 0] - e1[:, 0] * e2[:, 2],
                  e1[:, 0] * e2[:, 1] - e1[:, 1] * e2[:, 0]], axis=1)
    cc = c[:, 0] * c[:, 0] + c[:, 1] * c[:, 1] + c[:, 2] * c[:, 2]
    used = cc != 0.0
    with np.errstate(all="ignore"):
        ln = np.sqrt(cc)
        w = ln * 0.5
        n = c / ln[:, None]
        d = -(n[:, 0] * q0[:, 0] + n[:, 1] * q0[:, 1] + n[:, 2] * q0[:, 2])
        wn = w[:, None] * n
        A = np.stack([wn[:, 0] * n[:, 0], wn[:, 0] * n[:, 1], wn[:, 0] * n[:, 2], wn[:, 1] * n[:, 1],
                      wn[:, 1] * n[:, 2], wn[:, 2] * n[:, 2]], axis=1)
        b = (w * d)[:, None] * n
    A[~used] = 0.0
    b[~used] = 0.0
    return A, b, used


def quadric_solve(A: np.ndarray, b: np.ndarray):
    """-> (x [k, 3] translated, ok [k], det [k], trace [k]) with the spec's cofactor formulas."""
    a00, a01, a02, a11, a12, a22 = (A[:, i] for i in range(6))
    c00 = a11 * a22 - a12 * a12
    c01 = a02 * a12 - a01 * a22
    c02 = a01 * a12 - a02 * a11
    c11 = a00 * a22 - a02 * a02
    c12 = a01 * a02 - a00 * a12
    c22 = a00 * a11 - a01 * a01
    det = (a00 * c00 + a01 * c01) + a02 * c02
    tr = (a00 + a11) + a22
    ok = (tr > 0.0) & (det > DET_REL * tr * tr * tr)
    with np.errstate(all="ignore"):
        x = -np.stack([(c00 * b[:, 0] + c01 * b[:, 1]) + c02 * b[:, 2],
                       (c01 * b[:, 0] + c11 * b[:, 1]) + c12 * b[:, 2],
                       (c02 * b[:, 0] + c12 * b[:, 1]) + c22 * b[:, 2]], axis=1) / det[:, None]
    return x, ok, det, tr


def _canonical(ct: np.ndarray):
    """Rotation of every [T, 3] id triple that starts at its smallest id."""
    r = np.argmin(ct, axis=1)
    i = np.arange(len(ct))
    return np.stack([ct[i, r], ct[i, (r + 1) % 3], ct[i, (r + 2) % 3]], axis=1)


class Detail(dict):
    """Per-cluster intermediate values for the tolerance and branch checks of the tests."""


def simplify_mesh(mesh, voxel_size: float, contraction: str = "average", detail: Optional[Detail] = None) -> Mesh:
    """Vectorised restatement of the spec (module docstring)."""
    vs, v, c, t, nrm, rows = _check(mesh, voxel_size, contraction)
    V = len(v)
    if V == 0:
        return Mesh(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int32),
                    None if nrm is None else np.zeros((0, 3)), np.zeros(0, np.int64))
    idx, bmin, vmin = cluster_index(v, vs)
    cid, rep = _clusters(idx)
    k = len(rep)
    p = v.astype(F64)
    avg = _exact_sums(p, cid, k, 24, True)
    col = _exact_sums(c.astype(F64), cid, k, 24, True).astype(np.float32)
    pos = avg.astype(np.float32)
    if contraction == "quadric":
        A, b, _ = triangle_quadrics(p - bmin[None, :], t)
        QA, Qb = np.zeros((k, 6)), np.zeros((k, 3))
        corner = cid[t].reshape(-1)                     # (triangle, corner) order
        np.add.at(QA, corner, np.repeat(A, 3, axis=0))
        np.add.at(Qb, corner, np.repeat(b, 3, axis=0))
        x, ok, det, tr = quadric_solve(QA, Qb)
        x = x + bmin[None, :]
        cidx = idx[rep]
        lo, hi = vmin[None, :] + cidx * vs, vmin[None, :] + (cidx + 1) * vs
        with np.errstate(invalid="ignore"):
            inside = ((x >= lo) & (x <= hi)).all(axis=1)
        use = ok & inside
        pos[use] = x[use].astype(np.float32)
        if detail is not None:
            detail.update(A=QA, b=Qb, det=det, trace=tr, x=x, lo=lo, hi=hi, quadric=use)
    normals = None
    if nrm is not None:
        normals = _normalise(_exact_sums(nrm, cid, k, 53, False))
    if detail is not None:
        detail.update(count=np.bincount(cid, minlength=k), bmin=bmin, vmin=vmin, cid=cid)
    if len(t):
        ct = cid[t]
        keep = (ct[:, 0] != ct[:, 1]) & (ct[:, 1] != ct[:, 2]) & (ct[:, 0] != ct[:, 2])
        can = _canonical(ct[keep])
        if len(can):
            _, first = np.unique(can, axis=0, return_index=True)   # first occurrence of every canonical form
            tris = can[np.sort(first)].astype(np.int32)
        else:
            tris = np.zeros((0, 3), np.int32)
    else:
        tris = np.zeros((0, 3), np.int32)
    return Mesh(pos, col, tris, normals, rows[rep])


def simplify_mesh_loop(mesh, voxel_size: float, contraction: str = "average") -> Mesh:
    """Per-cluster / per-triangle loop over Python numbers, with rational sums: the second restatement."""
    vs, v, c, t, nrm, rows = _check(mesh, voxel_size, contraction)
    V = len(v)
    if V == 0:
        return Mesh(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int32),
                    None if nrm is None else np.zeros((0, 3)), np.zeros(0, np.int64))
    P = [tuple(float(a) for a in row) for row in v]
    bmin = [min(p[k] for p in P) for k in range(3)]
    vmin = [bmin[k] - vs * 0.5 for k in range(3)]
    idx = [tuple(math.floor((p[k] - vmin[k]) / vs) for k in range(3)) for p in P]
    if max(max(i) for i in idx) >= (1 << VOXEL_INDEX_BITS):
        raise ValueError("voxel_size is too small.")
    ids, members = {}, []
    for i, key in enumerate(idx):                      # first sight = lowest member id
        if key not in ids:
            ids[key] = len(members)
            members.append([])
        members[ids[key]].append(i)
    cid = [ids[key] for key in idx]
    pos, col, out_nrm = [], [], []
    for mem in members:
        n = len(mem)
        pos.append([float(sum((Fraction(P[i][k]) for i in mem), Fraction(0)) / n) for k in range(3)])
        col.append([float(sum((Fraction(float(c[i][k])) for i in mem), Fraction(0)) / n) for k in range(3)])
        if nrm is not None:
            s = [float(sum((Fraction(float(nrm[i][k])) for i in mem), Fraction(0))) for k in range(3)]
            nn = s[0] * s[0] + s[1] * s[1] + s[2] * s[2]
            out_nrm.append([0.0, 0.0, 0.0] if nn == 0.0 else [s[k] / math.sqrt(nn) for k in range(3)])
    if contraction == "quadric":
        QA = [[0.0] * 6 for _ in members]
        Qb = [[0.0] * 3 for _ in members]
        for tri in t:
            q = [[P[int(j)][k] - bmin[k] for k in range(3)] for j in tri]
            e1 = [q[1][k] - q[0][k] for k in range(3)]
            e2 = [q[2][k] - q[0][k] for k in range(3)]
            cr = [e1[1] * e2[2] - e1[2] * e2[1], e1[2] * e2[0] - e1[0] * e2[2], e1[0] * e2[1] - e1[1] * e2[0]]
            cc = cr[0] * cr[0] + cr[1] * cr[1] + cr[2] * cr[2]
            if cc == 0.0:
                continue
            ln = math.sqrt(cc)
            w = ln * 0.5
            nv = [cr[k] / ln for k in range(3)]
            d = -(nv[0] * q[0][0] + nv[1] * q[0][1] + nv[2] * q[0][2])
            wn = [w * nv[k] for k in range(3)]
            a = [wn[0] * nv[0], wn[0] * nv[1], wn[0] * nv[2], wn[1] * nv[1], wn[1] * nv[2], wn[2] * nv[2]]
            bb = [(w * d) * nv[k] for k in range(3)]
            for j in tri:
                g = cid[int(j)]
                for k in range(6):
                    QA[g][k] += a[k]
                for k in range(3):
                    Qb[g][k] += bb[k]
        for g in range(len(members)):
            a00, a01, a02, a11, a12, a22 = QA[g]
            c00, c01, c02 = a11 * a22 - a12 * a12, a02 * a12 - a01 * a22, a01 * a12 - a02 * a11
            c11, c12, c22 = a00 * a22 - a02 * a02, a01 * a02 - a00 * a12, a00 * a11 - a01 * a01
            det = (a00 * c00 + a01 * c01) + a02 * c02
            tr = (a00 + a11) + a22
            if not (tr > 0.0 and det > DET_REL * tr * tr * tr):
                continue
            b0, b1, b2 = Qb[g]
            x = [-((c00 * b0 + c01 * b1) + c02 * b2) / det + bmin[0],
                 -((c01 * b0 + c11 * b1) + c12 * b2) / det + bmin[1],
                 -((c02 * b0 + c12 * b1) + c22 * b2) / det + bmin[2]]
            key = idx[members[g][0]]
            if all(vmin[k] + key[k] * vs <= x[k] <= vmin[k] + (key[k] + 1) * vs for k in range(3)):
                pos[g] = x
    seen, tris = set(), []
    for tri in t:
        a, b, cc = (cid[int(j)] for j in tri)
        if a == b or b == cc or a == cc:
            continue
        m = min(a, b, cc)
        can = (a, b, cc) if m == a else ((b, cc, a) if m == b else (cc, a, b))
        if can not in seen:
            seen.add(can)
            tris.append(can)
    rep = [mem[0] for mem in members]
    return Mesh(np.array(pos, F64).astype(np.float32).reshape(-1, 3), np.array(col, F64).astype(np.float32).reshape(-1, 3),
                np.array(tris, np.int32).reshape(-1, 3), None if nrm is None else np.array(out_nrm, F64).reshape(-1, 3),
                rows[np.array(rep, np.int64)])
