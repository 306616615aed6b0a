"""Row f5: density clustering of a point cloud, Open3D ``PointCloud::ClusterDBSCAN`` and
``PointCloud::RemoveRadiusOutliers`` (geometry/PointCloud.cpp).  PARITY UNPINNED: Open3D is not installed here; this
restates its published source.

Points are float32 [N, 3] taken as float64.  Point j is a neighbour of point i when d2(i, j) < eps * eps (strict:
nanoflann's radius result set), d2 = (xi - xj)^2 + (yi - yj)^2 + (zi - zj)^2 summed left to right in float64 with no
contraction; the point itself is a neighbour.

* ``remove_radius_outlier``: row i is kept iff |N(i)| > nb_points, kept rows in input order.
* ``cluster_dbscan``: a point is core iff |N(i)| >= min_points.  Clusters are the connected components of the cores
  under the neighbour relation, numbered 0, 1, ... in increasing order of their lowest core index.  A non-core point
  takes the smallest cluster id among its core neighbours, else -1.

Why this is Open3D's result, which visits points in BFS order: its outer loop seeds a cluster only at an unlabelled
core point, and that seed is the lowest core of its component (a lower core of the same component would have seeded
the cluster earlier and its BFS would have labelled this point).  The BFS expands only cores, so a cluster is exactly
a core component.  A non-core point is labelled by the first cluster whose BFS reaches it, the lowest-numbered
cluster with a core within eps; the -1 an earlier outer-loop visit wrote is overwritten.

Two forms: ``cluster_dbscan`` (cKDTree candidates, d2 recomputed and filtered exactly, scipy connected components)
and ``cluster_dbscan_loop`` (Open3D's loop over precomputed neighbour lists, small clouds only).

The device grid has cells of side eps / 2 * (1 + 2^-20) and refuses a cloud whose bounding box needs 1048574 cells
or more along an axis (``grid_fits``); the checks below raise the same ValueError.
"""
from __future__ import annotations

import math

import numpy as np

F64 = np.float64
GRID_CELL_LIMIT = 1048574.0
RADIUS_MESSAGE = "Illegal input parameters, number of points and radius must be positive"


def cell_size(eps: float) -> float:
    return eps * 0.5 * (1.0 + 2.0 ** -20)


def check_eps(eps, name: str = "eps") -> float:
    e = float(eps)
    if not (math.isfinite(e) and e > 0.0 and 0.0 < e * e < math.inf):
        raise ValueError(f"{name} must be a finite positive number")
    return e


def check_min_points(min_points) -> int:
    k = int(min_points)
    if k != min_points or k < 0:
        raise ValueError("min_points must be an integer >= 0")
    return k


def grid_fits(points: np.ndarray, eps: float) -> bool:
    """The device grid holds the cloud: every axis of its float32 bounding box spans fewer than 1048574 cells."""
    p = np.asarray(points, dtype=np.float32)
    if len(p) == 0:
        return True
    lo, hi = p.min(axis=0).astype(F64), p.max(axis=0).astype(F64)
    cs = cell_size(eps)
    return all((h - l if h > l else 0.0) / cs < GRID_CELL_LIMIT for l, h in zip(lo, hi))


def check_points(points: np.ndarray, eps: float) -> np.ndarray:
    p = np.ascontiguousarray(points, dtype=np.float32)
    if p.ndim != 2 or p.shape[1] != 3:
        raise ValueError("points must be float32 [N, 3]")
    if not np.isfinite(p).all():
        raise ValueError("points must be finite")
    if not grid_fits(p, eps):
        raise ValueError(f"eps {eps!r} is too small for the extent of the cloud: the grid holds fewer than "
                         f"{int(GRID_CELL_LIMIT)} cells of side eps / 2 per axis")
    return p


def _d2(p: np.ndarray, i: np.ndarray, j: np.ndarray) -> np.ndarray:
    d2 = (p[i, 0] - p[j, 0]) * (p[i, 0] - p[j, 0])
    d2 += (p[i, 1] - p[j, 1]) * (p[i, 1] - p[j, 1])
    d2 += (p[i, 2] - p[j, 2]) * (p[i, 2] - p[j, 2])
    return d2


def neighbour_pairs(points: np.ndarray, eps: float, chunk: int = 1 << 24):
    """Every unordered pair i < j of distinct rows with d2 < eps * eps: (i int64 [P], j int64 [P])."""
    from scipy.spatial import cKDTree
    p = np.ascontiguousarray(points, dtype=F64)
    if len(p) < 2:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    pairs = cKDTree(p).query_pairs(eps * (1.0 + 1e-9), output_type="ndarray")
    e2 = eps * eps
    keep_i, keep_j = [np.zeros(0, np.int64)], [np.zeros(0, np.int64)]
    for s in range(0, len(pairs), chunk):
        c = pairs[s:s + chunk]
        i, j = c[:, 0].astype(np.int64), c[:, 1].astype(np.int64)
        ok = _d2(p, i, j) < e2
        keep_i.append(i[ok])
        keep_j.append(j[ok])
    del pairs
    return np.concatenate(keep_i), np.concatenate(keep_j)


def neighbour_counts(n: int, i: np.ndarray, j: np.ndarray) -> np.ndarray:
    return 1 + np.bincount(i, minlength=n) + np.bincount(j, minlength=n)


def _labels(n: int, i: np.ndarray, j: np.ndarray, min_points: int) -> np.ndarray:
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    core = neighbour_counts(n, i, j) >= min_points
    cc = core[i] & core[j]
    g = coo_matrix((np.ones(int(cc.sum()), np.int8), (i[cc], j[cc])), shape=(n, n)).tocsr()
    _, comp = connected_components(g, directed=False)
    labels = np.full(n, -1, np.int32)
    cores = np.nonzero(core)[0]
    if len(cores):
        # clusters in increasing order of their lowest core: the components in order of first appearance among cores
        first, pos = np.unique(comp[cores], return_index=True)
        order = np.argsort(pos, kind="stable")
        rank = np.empty(len(first), np.int32)
        rank[order] = np.arange(len(first), dtype=np.int32)
        labels[cores] = rank[np.searchsorted(first, comp[cores])]
    # a non-core point: the smallest cluster among its core neighbours
    big = np.iinfo(np.int32).max
    border = np.full(n, big, np.int64)
    for a, b in ((i, j), (j, i)):
        sel = ~core[a] & core[b]
        np.minimum.at(border, a[sel], labels[b[sel]].astype(np.int64))
    nc = ~core & (border < big)
    labels[nc] = border[nc].astype(np.int32)
    return labels


def cluster_dbscan(points: np.ndarray, eps: float, min_points: int) -> np.ndarray:
    """``np.asarray(pcd.cluster_dbscan(eps, min_points))``: int32 [N] labels."""
    eps, min_points = check_eps(eps), check_min_points(min_points)
    p = check_points(points, eps)
    n = len(p)
    if n == 0:
        return np.zeros(0, np.int32)
    i, j = neighbour_pairs(p, eps)
    return _labels(n, i, j, min_points)


def cluster_sizes(labels: np.ndarray) -> np.ndarray:
    """Points of every cluster, uint32 [K]."""
    k = int(labels.max()) + 1 if len(labels) else 0
    return np.bincount(labels[labels >= 0], minlength=k).astype(np.uint32)


def remove_small_clusters(points: np.ndarray, eps: float, min_points: int, min_size: int = 1):
    """Rows of clusters of at least min_size points, in input order: (kept index int64, labels int32, sizes uint32)."""
    labels = cluster_dbscan(points, eps, min_points)
    sizes = cluster_sizes(labels)
    keep = labels >= 0
    keep[keep] = sizes[labels[keep]] >= min_size
    return np.nonzero(keep)[0].astype(np.int64), labels, sizes


def remove_radius_outlier(points: np.ndarray, nb_points: int, radius: float) -> np.ndarray:
    """Open3D ``RemoveRadiusOutliers``: kept index int64, rows with more than nb_points neighbours (itself counted)."""
    r = float(radius)
    if int(nb_points) < 1 or not (math.isfinite(r) and r > 0.0 and 0.0 < r * r < math.inf):
        raise ValueError(RADIUS_MESSAGE)
    p = check_points(points, r)
    i, j = neighbour_pairs(p, r)
    return np.nonzero(neighbour_counts(len(p), i, j) > int(nb_points))[0].astype(np.int64)


# ---- literal forms, small clouds only ----------------------------------------------------------------------------
def neighbour_lists(points: np.ndarray, eps: float):
    """Brute force: the neighbours of every point, itself included, ascending."""
    p = np.ascontiguousarray(points, dtype=F64)
    n = len(p)
    ii, jj = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    near = _d2(p, ii.ravel(), jj.ravel()).reshape(n, n) < eps * eps
    return [np.nonzero(near[k])[0].tolist() for k in range(n)]


def cluster_dbscan_loop(points: np.ndarray, eps: float, min_points: int) -> np.ndarray:
    """Open3D's ClusterDBSCAN loop over precomputed neighbour lists (-2 = not yet visited)."""
    nbs_all = neighbour_lists(points, eps)
    n = len(nbs_all)
    labels = [-2] * n
    cluster_label = 0
    for idx in range(n):
        if labels[idx] != -2:
            continue
        nbs = nbs_all[idx]
        if len(nbs) < min_points:
            labels[idx] = -1
            continue
        nbs_next = list(dict.fromkeys(nbs))   # Open3D iterates an unordered_set: the order does not change the result
        nbs_visited = {idx}
        labels[idx] = cluster_label
        while nbs_next:
            nb = nbs_next.pop(0)
            nbs_visited.add(nb)
            if labels[nb] == -1:
                labels[nb] = cluster_label
            if labels[nb] != -2:
                continue
            labels[nb] = cluster_label
            if len(nbs_all[nb]) >= min_points:
                for qnb in nbs_all[nb]:
                    if qnb not in nbs_visited and qnb not in nbs_next:
                        nbs_next.append(qnb)
        cluster_label += 1
    return np.asarray(labels, np.int32)


def remove_radius_outlier_brute(points: np.ndarray, nb_points: int, radius: float) -> np.ndarray:
    nbs = neighbour_lists(points, radius)
    return np.asarray([k for k, x in enumerate(nbs) if len(x) > nb_points], np.int64)
