"""TEST INFRASTRUCTURE ONLY -- CPU oracle for the connected components of a triangle mesh and the removal of
triangles by a mask (DESIGN row m3).

SPEC FROZEN HERE, NO REFERENCE CODE: the reference leaves mesh clean-up to Open3D (backend/app.py:271-308).  This
restates Open3D's ``TriangleMesh::ClusterConnectedTriangles``, ``RemoveTrianglesByMask`` and
``RemoveUnreferencedVertices`` (geometry/TriangleMesh.cpp), with a fixed-point cluster area where Open3D sums in BFS
order; Open3D is not installed in the build container, so parity is UNPINNED.  The product package never imports
this module.

Input: a mesh in the ``TriangleMesh`` layout (vertices f32 [V, 3], colors f32 [V, 3], triangles i32 [T, 3],
vertex_normals f64 [V, 3] or None, vertex_rows i64 [V]).

  errors        a triangle id < 0 or >= V; a vertex with a non-finite coordinate (ValueError)
  connectivity  two triangles are connected when they share an edge, an unordered vertex pair (Open3D's
                ``GetEdgeToTrianglesMap``): sharing only a vertex does not connect; a non-manifold edge connects every
                triangle on it; (a, a, b) has the edges {a,a}, {a,b}, {a,b}; repeated triangles are connected
  numbering     clusters in ascending order of their lowest triangle (the order in which Open3D's BFS, started at
                the lowest unvisited triangle, assigns them; independent of the order it visits neighbours)
  area          per triangle Open3D's ``GetTriangleArea`` in float64 from the float32 vertices: x = p0 - p1,
                y = p0 - p2, c = x cross y (Eigen's order), 0.5 * sqrt((c0*c0 + c1*c1) + c2*c2)
  cluster area  s = 2^(62 - e_a - e_T) with max_t a_t < 2^e_a (frexp; 0 when every area is 0) and T <= 2^e_T;
                q_t = rint(a_t s) (half to even, exact integers); area = float64(sum of q_t) / s, rounded once
  outputs       triangle_clusters int32 [T], cluster_n_triangles int64 [K], cluster_area float64 [K]
  removal       ``remove_triangles_by_mask(mesh, mask)`` drops the triangles where mask is True, keeping the others
                in input order; with remove_unreferenced only vertices a kept triangle uses stay, in input order,
                with their colours, normals and rows unchanged, and the triangles are remapped to the new ids

Two restatements of the clustering: ``cluster_connected_triangles`` (scipy's connected_components on the
triangle-edge graph, relabelled by lowest triangle) and ``cluster_connected_triangles_loop`` (Open3D's BFS per
triangle), which the CPU tests check against each other.
"""
from __future__ import annotations

import math
from collections import deque
from typing import Optional

import numpy as np
import scipy.sparse as sp
from scipy.sparse.csgraph import connected_components

from .d2pc_mesh_oracle import Mesh
from .d2pc_oracle import F64


def check_mesh(mesh):
    """(float32 vertices [V, 3], int64 triangles [T, 3]); ValueError for a bad id or a non-finite vertex."""
    v = np.asarray(mesh.vertices, np.float32).reshape(-1, 3)
    t = np.asarray(mesh.triangles).reshape(-1, 3).astype(np.int64)
    if len(t) and (t.min() < 0 or t.max() >= len(v)):
        raise ValueError("a triangle refers to a vertex that does not exist")
    if not np.isfinite(v).all():
        raise ValueError("the mesh has a non-finite vertex coordinate")
    return v, t


def triangle_areas(v: np.ndarray, t: np.ndarray) -> np.ndarray:
    """Open3D's GetTriangleArea of every triangle, float64."""
    p = v.astype(F64)
    p0, p1, p2 = p[t[:, 0]], p[t[:, 1]], p[t[:, 2]]
    x, y = p0 - p1, p0 - p2
    c0 = x[:, 1] * y[:, 2] - x[:, 2] * y[:, 1]
    c1 = x[:, 2] * y[:, 0] - x[:, 0] * y[:, 2]
    c2 = x[:, 0] * y[:, 1] - x[:, 1] * y[:, 0]
    return 0.5 * np.sqrt((c0 * c0 + c1 * c1) + c2 * c2)


def area_scale(areas: np.ndarray) -> float:
    """s = 2^(62 - e_a - e_T) of the fixed-point cluster areas."""
    T = len(areas)
    amax = float(areas.max()) if T else 0.0
    ea = math.frexp(amax)[1] if amax > 0.0 else 0
    et = (T - 1).bit_length() if T > 1 else 0
    return math.ldexp(1.0, 62 - ea - et)


def area_terms(areas: np.ndarray, s: float) -> np.ndarray:
    """q_t = rint(a_t s) as int64 (a_t s is exact: s is a power of two; every q_t < 2^62)."""
    return np.rint(areas * s).astype(np.int64)


def _finish_areas(sums, s: float) -> np.ndarray:
    return np.array([float(int(x)) / s for x in sums], dtype=F64)


def _edge_keys(t: np.ndarray) -> np.ndarray:
    """[T, 3] keys (min << 32) | max of the edges (t0, t1), (t1, t2), (t2, t0)."""
    a = t
    b = np.roll(t, -1, axis=1)
    return (np.minimum(a, b) << 32) | np.maximum(a, b)


def cluster_connected_triangles(mesh):
    """(triangle_clusters int32 [T], cluster_n_triangles int64 [K], cluster_area float64 [K]), vectorised."""
    v, t = check_mesh(mesh)
    T = len(t)
    if T == 0:
        return np.zeros(0, np.int32), np.zeros(0, np.int64), np.zeros(0, F64)
    _, eid = np.unique(_edge_keys(t).reshape(-1), return_inverse=True)
    E = int(eid.max()) + 1
    rows = np.repeat(np.arange(T), 3)
    g = sp.coo_matrix((np.ones(3 * T, np.int8), (rows, T + eid.reshape(-1))), shape=(T + E, T + E)).tocsr()
    _, lab = connected_components(g, directed=False)
    lab = lab[:T]
    comps, first = np.unique(lab, return_index=True)
    order = np.argsort(first, kind="stable")         # by lowest triangle
    rank = np.empty(len(comps), np.int64)
    rank[order] = np.arange(len(comps))
    remap = np.full(int(lab.max()) + 1, -1, np.int64)
    remap[comps] = rank
    clusters = remap[lab]
    K = len(comps)
    n = np.bincount(clusters, minlength=K).astype(np.int64)
    areas = triangle_areas(v, t)
    s = area_scale(areas)
    sums = np.zeros(K, np.int64)
    np.add.at(sums, clusters, area_terms(areas, s))   # < 2^62: exact in int64
    return clusters.astype(np.int32), n, _finish_areas(sums, s)


def cluster_connected_triangles_loop(mesh, rng: Optional[np.random.Generator] = None):
    """Open3D's ClusterConnectedTriangles: a BFS from every unvisited triangle in ascending order over the
    edge-to-triangles map; with ``rng`` each triangle's neighbours are visited in a random order.  Areas are summed as
    Python integers of the same fixed-point terms."""
    v, t = check_mesh(mesh)
    T = len(t)
    edge_tris = {}
    for i in range(T):
        a, b, c = (int(x) for x in t[i])
        for e0, e1 in ((a, b), (b, c), (c, a)):
            edge_tris.setdefault((min(e0, e1), max(e0, e1)), []).append(i)
    areas = triangle_areas(v, t) if T else np.zeros(0)
    s = area_scale(areas)
    q = [int(x) for x in area_terms(areas, s)]
    clusters = [-1] * T
    n_tri, sums = [], []
    for start in range(T):
        if clusters[start] != -1:
            continue
        cid = len(n_tri)
        clusters[start] = cid
        n, acc = 1, q[start]
        queue = deque([start])
        while queue:
            i = queue.popleft()
            a, b, c = (int(x) for x in t[i])
            nbs = []
            for e0, e1 in ((a, b), (b, c), (c, a)):
                nbs += edge_tris[(min(e0, e1), max(e0, e1))]
            if rng is not None:
                nbs = [nbs[k] for k in rng.permutation(len(nbs))]
            for j in nbs:
                if clusters[j] == -1:
                    clusters[j] = cid
                    n += 1
                    acc += q[j]
                    queue.append(j)
        n_tri.append(n)
        sums.append(acc)
    return np.array(clusters, np.int32), np.array(n_tri, np.int64), _finish_areas(sums, s)


def remove_triangles_by_mask(mesh, mask, remove_unreferenced: bool = True) -> Mesh:
    """Open3D's remove_triangles_by_mask (mask True: the triangle goes), then remove_unreferenced_vertices."""
    v, t = check_mesh(mesh)
    mask = np.asarray(mask, bool).reshape(-1)
    if len(mask) != len(t):
        raise ValueError("the mask must have one entry per triangle")
    kept = t[~mask]
    V = len(v)
    if remove_unreferenced:
        used = np.zeros(V, bool)
        used[kept.reshape(-1)] = True
    else:
        used = np.ones(V, bool)
    idx = np.nonzero(used)[0]
    newid = np.full(V, -1, np.int64)
    newid[idx] = np.arange(len(idx))
    nrm = mesh.vertex_normals
    return Mesh(v[idx], np.asarray(mesh.colors, np.float32).reshape(-1, 3)[idx],
                newid[kept].astype(np.int32).reshape(-1, 3),
                None if nrm is None else np.asarray(nrm, F64).reshape(-1, 3)[idx],
                np.asarray(mesh.vertex_rows, np.int64).reshape(-1)[idx])


def small_component_mask(mesh, min_triangles=None, min_area=None) -> np.ndarray:
    """True for every triangle of a cluster with fewer than ``min_triangles`` triangles or less area than
    ``min_area``."""
    clusters, n, area = cluster_connected_triangles(mesh)
    remove = np.zeros(len(clusters), bool)
    if min_triangles is not None:
        remove |= n[clusters] < min_triangles
    if min_area is not None:
        remove |= area[clusters] < min_area
    return remove


def remove_small_components(mesh, min_triangles=None, min_area=None) -> Mesh:
    return remove_triangles_by_mask(mesh, small_component_mask(mesh, min_triangles, min_area))
