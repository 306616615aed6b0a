"""TEST INFRASTRUCTURE ONLY -- CPU oracle for point normals (the first step of the reference's mesh builder,
backend/app.py:271-308, 508-535: Open3D ``estimate_normals``), and the PLY vertices of a cloud with normals.

PARITY UNPINNED: Open3D is not installed in the build container.  This restates its published source
(geometry/EstimateNormals.cpp, geometry/KDTreeFlann.cpp, io/file_format/FilePLY.cpp); the spec is frozen here,
as for statistical outlier removal, LAS and PLY in ``d2pc_oracle``.  The product package never imports it.
"""
from __future__ import annotations

from typing import Optional

import numpy as np

from .d2pc_oracle import F64, ply_records


# --------------------------------------------------------------------------------------------
# normals (the mesh builder's first step, backend/app.py:271-308: Open3D estimate_normals)
# --------------------------------------------------------------------------------------------
PLY_NORMAL_RECORD_DTYPE = np.dtype([("x", "<f8"), ("y", "<f8"), ("z", "<f8"), ("nx", "<f8"), ("ny", "<f8"),
                                    ("nz", "<f8"), ("red", "u1"), ("green", "u1"), ("blue", "u1")])
PLY_NORMAL_HEADER = ("ply\nformat binary_little_endian 1.0\ncomment Created by Open3D\nelement vertex {n}\n"
                     "property double x\nproperty double y\nproperty double z\n"
                     "property double nx\nproperty double ny\nproperty double nz\n"
                     "property uchar red\nproperty uchar green\nproperty uchar blue\nend_header\n")


def ply_normal_records(points: np.ndarray, normals: np.ndarray, colors: np.ndarray) -> np.ndarray:
    """Open3D's binary PLY vertices of a cloud with normals (its writer adds nx, ny, nz after z).  PARITY UNPINNED
    like ``ply_records``."""
    assert PLY_NORMAL_RECORD_DTYPE.itemsize == 51
    rec = np.zeros(len(points), dtype=PLY_NORMAL_RECORD_DTYPE)
    base = ply_records(points, colors)
    for f in ("x", "y", "z", "red", "green", "blue"):
        rec[f] = base[f]
    rec["nx"], rec["ny"], rec["nz"] = normals[:, 0], normals[:, 1], normals[:, 2]
    return rec


def _axiswise_d2(q: np.ndarray, p: np.ndarray) -> np.ndarray:
    """nanoflann's L2_Simple in float64: d2 = dx*dx; d2 += dy*dy; d2 += dz*dz (q [m,1,3], p [m,c,3])."""
    d = q - p
    d2 = d[..., 0] * d[..., 0]
    d2 = d2 + d[..., 1] * d[..., 1]
    d2 = d2 + d[..., 2] * d[..., 2]
    return d2


def _first_k(p, rows, cand, k, r2):
    """cand int64 [m, c] candidate rows (-1 = none) of the queries `rows` -> ([m, k] rows, [m, k] valid) in
    ascending (d2, row) order."""
    big = np.iinfo(np.int64).max
    ok = cand >= 0
    c = np.where(ok, cand, 0)
    d2 = np.where(ok, _axiswise_d2(p[rows][:, None, :], p[c]), np.inf)
    key_row = np.where(ok, cand, big)
    order = np.lexsort((key_row, d2), axis=1)[:, :k]
    d2s = np.take_along_axis(d2, order, axis=1)
    rs = np.take_along_axis(key_row, order, axis=1)
    if rs.shape[1] < k:  # fewer candidates than k (radius mode)
        pad = k - rs.shape[1]
        rs = np.concatenate([rs, np.full((len(rs), pad), big)], axis=1)
        d2s = np.concatenate([d2s, np.full((len(d2s), pad), np.inf)], axis=1)
    valid = d2s < r2
    return np.where(valid, rs, 0), valid


def neighbours(points: np.ndarray, knn: int = 30, radius: Optional[float] = None, workers: int = 1):
    """Each point's neighbourhood as the normals use it: the knn nearest points (itself included), with a radius
    only those with d2 < radius^2 (strict, as nanoflann's radius result set), ties ordered by (d2, source row).
    Exact: scipy's k-th distance, every candidate up to a hair above it, d2 recomputed axis by axis in float64,
    sorted by (d2, row).  Returns (rows int64 [N, k], valid bool [N, k]) in ascending order, k = min(knn, N).
    ``workers`` is scipy's thread count for the tree queries (-1: all cores)."""
    from scipy.spatial import cKDTree
    p = np.ascontiguousarray(points, dtype=F64)
    n = len(p)
    k = min(int(knn), n)
    if n == 0:
        return np.zeros((0, 0), np.int64), np.zeros((0, 0), bool)
    r2 = float(radius) * float(radius) if radius is not None and radius > 0 else np.inf
    tree = cKDTree(p)
    kq = min(n, k + 16)
    dist, idx = tree.query(p, k=kq, workers=workers)
    dist, idx = dist.reshape(n, kq), idx.reshape(n, kq).astype(np.int64)
    lim = dist[:, k - 1]
    if r2 < np.inf:
        lim = np.minimum(lim, float(radius))
    hair = lim * (1.0 + 1e-9)
    # candidates: every point within the hair; when the kq-th returned point is still inside it, ask for all of them
    more = (dist[:, kq - 1] <= hair) if kq < n else np.zeros(n, bool)
    cand = np.where(dist <= hair[:, None], idx, -1)
    rows_out = np.zeros((n, k), np.int64)
    valid_out = np.zeros((n, k), bool)
    easy = np.nonzero(~more)[0]
    for s in range(0, len(easy), 65536):
        r = easy[s:s + 65536]
        rows_out[r], valid_out[r] = _first_k(p, r, cand[r], k, r2)
    hard = np.nonzero(more)[0]
    for s in range(0, len(hard), 2048):
        r = hard[s:s + 2048]
        lists = tree.query_ball_point(p[r], hair[r], workers=workers)
        width = max(len(x) for x in lists)
        c = np.full((len(r), width), -1, np.int64)
        for t, x in enumerate(lists):
            c[t, :len(x)] = x
        rows_out[r], valid_out[r] = _first_k(p, r, c, k, r2)
    return rows_out, valid_out


def covariances(points: np.ndarray, rows: np.ndarray, valid: np.ndarray) -> np.ndarray:
    """Open3D ``ComputeCovariance`` over each neighbourhood in the given order -> float64 [N, 6] =
    c00, c01, c02, c11, c12, c22; fewer than 3 neighbours -> identity (``EstimatePerPointCovariances``)."""
    p = np.ascontiguousarray(points, dtype=F64)
    n = len(p)
    cu = np.zeros((n, 9), F64)
    for t in range(rows.shape[1]):
        q = p[rows[:, t]]
        v = valid[:, t]
        terms = (q[:, 0], q[:, 1], q[:, 2], q[:, 0] * q[:, 0], q[:, 0] * q[:, 1], q[:, 0] * q[:, 2],
                 q[:, 1] * q[:, 1], q[:, 1] * q[:, 2], q[:, 2] * q[:, 2])
        for j, x in enumerate(terms):
            cu[:, j] = np.where(v, cu[:, j] + x, cu[:, j])
    cnt = valid.sum(axis=1)
    out = np.tile(np.array([1.0, 0.0, 0.0, 1.0, 0.0, 1.0]), (n, 1))
    ok = cnt >= 3
    c = cu[ok] / cnt[ok, None].astype(F64)
    out[ok, 0] = c[:, 3] - c[:, 0] * c[:, 0]
    out[ok, 3] = c[:, 6] - c[:, 1] * c[:, 1]
    out[ok, 5] = c[:, 8] - c[:, 2] * c[:, 2]
    out[ok, 1] = c[:, 4] - c[:, 0] * c[:, 1]
    out[ok, 2] = c[:, 5] - c[:, 0] * c[:, 2]
    out[ok, 4] = c[:, 7] - c[:, 1] * c[:, 2]
    return out


def _cross(a, b):
    return np.stack([a[:, 1] * b[:, 2] - a[:, 2] * b[:, 1], a[:, 2] * b[:, 0] - a[:, 0] * b[:, 2],
                     a[:, 0] * b[:, 1] - a[:, 1] * b[:, 0]], axis=1)


def _dot(a, b):
    return a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1] + a[:, 2] * b[:, 2]


def _eigenvector0(A, lam):
    """ComputeEigenvector0: the largest cross product of two rows of A - lam I, normalised."""
    a00, a01, a02, a11, a12, a22 = A.T
    r0 = np.stack([a00 - lam, a01, a02], 1)
    r1 = np.stack([a01, a11 - lam, a12], 1)
    r2 = np.stack([a02, a12, a22 - lam], 1)
    x01, x02, x12 = _cross(r0, r1), _cross(r0, r2), _cross(r1, r2)
    d0, d1, d2 = _dot(x01, x01), _dot(x02, x02), _dot(x12, x12)
    imax = np.zeros(len(A), np.int64)
    dmax = d0.copy()
    imax[d1 > dmax] = 1
    dmax = np.where(d1 > dmax, d1, dmax)
    imax[d2 > dmax] = 2
    v = np.where((imax == 0)[:, None], x01, np.where((imax == 1)[:, None], x02, x12))
    s = np.sqrt(np.where(imax == 0, d0, np.where(imax == 1, d1, d2)))
    return v / s[:, None]


def _eigenvector1(A, e0, lam):
    """ComputeEigenvector1: the eigenvector of lam inside the orthogonal complement of e0."""
    a00, a01, a02, a11, a12, a22 = A.T
    big = np.abs(e0[:, 0]) > np.abs(e0[:, 1])
    inv = np.where(big, 1 / np.sqrt(e0[:, 0] * e0[:, 0] + e0[:, 2] * e0[:, 2]),
                   1 / np.sqrt(e0[:, 1] * e0[:, 1] + e0[:, 2] * e0[:, 2]))
    zero = np.zeros(len(A))
    U = np.where(big[:, None], np.stack([-e0[:, 2] * inv, zero, e0[:, 0] * inv], 1),
                 np.stack([zero, e0[:, 2] * inv, -e0[:, 1] * inv], 1))
    V = _cross(e0, U)

    def mul(X):
        return np.stack([a00 * X[:, 0] + a01 * X[:, 1] + a02 * X[:, 2], a01 * X[:, 0] + a11 * X[:, 1] + a12 * X[:, 2],
                         a02 * X[:, 0] + a12 * X[:, 1] + a22 * X[:, 2]], 1)
    AU, AV = mul(U), mul(V)
    m00 = U[:, 0] * AU[:, 0] + U[:, 1] * AU[:, 1] + U[:, 2] * AU[:, 2] - lam
    m01 = U[:, 0] * AV[:, 0] + U[:, 1] * AV[:, 1] + U[:, 2] * AV[:, 2]
    m11 = V[:, 0] * AV[:, 0] + V[:, 1] * AV[:, 1] + V[:, 2] * AV[:, 2] - lam
    b00, b01, b11 = np.abs(m00), np.abs(m01), np.abs(m11)
    first = b00 >= b11
    mx = np.where(first, np.where(b00 < b01, b01, b00), np.where(b11 < b01, b01, b11))
    # absM00 >= absM11: rows (m00, m01); otherwise (m11, m01) -- the same two cases on (a, b) = (m_diag, m01)
    a = np.where(first, m00, m11)
    ba = np.where(first, b00, b11)
    t = np.where(ba >= b01, m01 / a, a / m01)            # the smaller over the larger
    s = 1 / np.sqrt(1 + t * t)
    big_a = ba >= b01
    ca = np.where(big_a, s, t * s)                       # new a (m00 or m11)
    cb = np.where(big_a, t * s, s)                       # new m01
    vec = np.where(first[:, None], cb[:, None] * U - ca[:, None] * V, ca[:, None] * U - cb[:, None] * V)
    return np.where((mx > 0)[:, None], vec, U)


def fast_eigen3x3(cov6: np.ndarray) -> np.ndarray:
    """Open3D's ``FastEigen3x3`` (Geometric Tools' robust 3x3 symmetric solver) on [N, 6] upper triangles ->
    [N, 3] eigenvector of the smallest eigenvalue as the solver returns it (the zero vector when max(C) == 0)."""
    C = np.ascontiguousarray(cov6, dtype=F64).reshape(-1, 6)
    n = len(C)
    mxc = C.max(axis=1) if n else np.zeros(0)
    out = np.zeros((n, 3))
    with np.errstate(all="ignore"):
        A = C / mxc[:, None]
        a00, a01, a02, a11, a12, a22 = A.T
        norm = a01 * a01 + a02 * a02 + a12 * a12
        q = (a00 + a11 + a22) / 3
        b00, b11, b22 = a00 - q, a11 - q, a22 - q
        p = np.sqrt((b00 * b00 + b11 * b11 + b22 * b22 + norm * 2) / 6)
        c00 = b11 * b22 - a12 * a12
        c01 = a01 * b22 - a12 * a02
        c02 = a01 * a12 - b11 * a02
        det = (b00 * c00 - a01 * c01 + a02 * c02) / (p * p * p)
        half = det * 0.5
        half = np.where(half < -1.0, -1.0, half)
        half = np.where(1.0 < half, 1.0, half)
        angle = np.arccos(half) / 3.0
        beta2 = np.cos(angle) * 2
        beta0 = np.cos(angle + 2.09439510239319549) * 2
        beta1 = -(beta0 + beta2)
        e0, e1, e2 = q + p * beta0, q + p * beta1, q + p * beta2
        pos = half >= 0
        v_first = _eigenvector0(A, np.where(pos, e2, e0))          # evec2 if half_det >= 0 else evec0
        first_min = np.where(pos, (e2 < e0) & (e2 < e1), (e0 < e1) & (e0 < e2))
        v_mid = _eigenvector1(A, v_first, e1)
        mid_min = (e1 < e0) & (e1 < e2)
        v_last = np.where(pos[:, None], _cross(v_mid, v_first), _cross(v_first, v_mid))
        res = np.where(first_min[:, None], v_first, np.where(mid_min[:, None], v_mid, v_last))
        d = A[:, [0, 3, 5]] * mxc[:, None]                          # A *= max_coeff, then the diagonal
        diag = np.tile([0.0, 0.0, 1.0], (n, 1))
        diag[(d[:, 1] < d[:, 0]) & (d[:, 1] < d[:, 2])] = [0.0, 1.0, 0.0]
        diag[(d[:, 0] < d[:, 1]) & (d[:, 0] < d[:, 2])] = [1.0, 0.0, 0.0]
        out = np.where((norm > 0)[:, None], res, diag)
    out[mxc == 0] = 0.0
    return out


def estimate_normals(points: np.ndarray, knn: int = 30, radius: Optional[float] = None,
                     orient_towards=(0.0, 0.0, 0.0), return_covariances: bool = False, workers: int = 1):
    """Open3D ``PointCloud::EstimateNormals(KDTreeSearchParamKNN(knn))`` -- or ``KDTreeSearchParamHybrid(radius,
    knn)`` when ``radius`` is given -- with ``fast_normal_computation=True`` on a cloud without normals, then
    ``OrientNormalsTowardsCameraLocation(orient_towards)`` (skipped when it is None).  Points are float32 taken as
    float64 (``Vector3dVector``).
    PARITY UNPINNED: Open3D is not installed in the build container; this restates its published source
    (geometry/EstimateNormals.cpp): neighbourhoods as ``neighbours`` (the (d2, row) tie rule is ours), covariance
    as ``covariances``, ``FastEigen3x3``, the result normalised and a zero vector replaced by (0, 0, 1); a normal is
    flipped where n . (c - p) < 0 (a product of exactly 0 keeps it).
    Returns float64 [N, 3] (and [N, 6] upper-triangle covariances when ``return_covariances``)."""
    p = np.ascontiguousarray(points, dtype=F64).reshape(-1, 3)
    if not np.isfinite(p).all():
        raise ValueError("estimate_normals: non-finite coordinates")
    rows, valid = neighbours(p, knn, radius, workers)
    cov = covariances(p, rows, valid)
    v = fast_eigen3x3(cov)
    s = _dot(v, v)
    zero = s == 0.0
    with np.errstate(all="ignore"):
        nrm = v / np.sqrt(s)[:, None]
    nrm[zero] = [0.0, 0.0, 1.0]
    if orient_towards is not None:
        ref = np.asarray(orient_towards, F64)[None, :] - p
        flip = _dot(nrm, ref) < 0.0
        nrm[flip] = nrm[flip] * -1.0
    return (nrm, cov) if return_covariances else nrm
