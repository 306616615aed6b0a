"""Meshes and the device-against-oracle comparison for mesh components (row m3), shared by
tests/test_components_cpu.py, tests/test_components_gpu.py and profiles/fuzz_components.py.

What must match exactly: triangle_clusters, cluster_n_triangles and the fixed-point cluster_area (bit for bit).
The areas are also held to their meaning: within n_c / (2 s) plus one float64 rounding of math.fsum of the
cluster's triangle areas.
"""
from __future__ import annotations

import math

import numpy as np

from oracle import d2pc_components_oracle as CO
from oracle import d2pc_mesh_oracle as MO


def mesh_of(xyz, tri, normals=False, seed=0):
    xyz = np.asarray(xyz, np.float32).reshape(-1, 3)
    V = len(xyz)
    rng = np.random.default_rng(seed)
    nrm = None
    if normals:
        nrm = rng.normal(size=(V, 3))
        nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    return MO.Mesh(xyz, rng.integers(0, 256, (V, 3)).astype(np.float32), np.asarray(tri, np.int32).reshape(-1, 3),
                   nrm, rng.permutation(10 * max(V, 1))[:V].astype(np.int64))


def hand_meshes():
    """name -> (mesh, expected triangle_clusters)."""
    sq = [[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0], [2, 0, 0], [2, 1, 0], [5, 5, 5], [6, 5, 5], [5, 6, 5]]
    fan = [[0, 0, 0], [0, 0, 1]] + [[math.cos(a), math.sin(a), 0.5] for a in np.linspace(0, 6, 5)]
    return {
        "shared edge": (mesh_of(sq, [[0, 1, 2], [1, 3, 2]]), [0, 0]),
        "shared vertex only": (mesh_of(sq, [[0, 1, 2], [1, 4, 5]]), [0, 1]),
        "non-manifold fan": (mesh_of(fan, [[0, 1, k] for k in range(2, 7)]), [0] * 5),
        "degenerate": (mesh_of(sq, [[0, 0, 1], [1, 0, 3], [4, 4, 4], [4, 4, 5], [5, 4, 6]]), [0, 0, 1, 1, 1]),
        "repeated": (mesh_of(sq, [[6, 7, 8], [0, 1, 2], [6, 7, 8], [8, 6, 7], [2, 1, 0]]), [0, 1, 0, 0, 1]),
        "unreferenced vertices": (mesh_of(sq, [[6, 7, 8], [3, 4, 5]]), [0, 1]),
        "chain by order": (mesh_of(sq, [[4, 5, 3], [0, 1, 2], [1, 3, 2], [3, 1, 4]]), [0, 0, 0, 0]),
        "empty": (mesh_of(sq, np.zeros((0, 3))), []),
        "no vertices": (mesh_of(np.zeros((0, 3)), np.zeros((0, 3))), []),
    }


def soup(rng, V, T, normals=False):
    """Random triangles over few vertices (many shared edges, non-manifold ones, degenerate and repeated triangles)."""
    xyz = (rng.random((V, 3)) * float(rng.choice([0.01, 1.0, 300.0])) + rng.normal(0, 5, 3)).astype(np.float32)
    tri = rng.integers(0, max(V, 1), (T, 3))
    if T and rng.random() < 0.5:
        k = T // 4
        tri[rng.integers(0, T, k)] = tri[rng.integers(0, T, k)]
    return mesh_of(xyz, tri, normals, int(rng.integers(1 << 30)))


def shuffled(mesh, rng):
    """The same mesh with its vertices and triangles in a random order."""
    V, T = len(mesh.vertices), len(mesh.triangles)
    pv, pt = rng.permutation(V), rng.permutation(T)
    inv = np.empty(V, np.int64)
    inv[pv] = np.arange(V)
    nrm = None if mesh.vertex_normals is None else mesh.vertex_normals[pv]
    return MO.Mesh(mesh.vertices[pv], mesh.colors[pv], inv[mesh.triangles[pt]].astype(np.int32), nrm,
                   mesh.vertex_rows[pv])


def strip(n, reverse=True):
    """A strip of n triangles, one component, in reversed order: every union hooks a long chain."""
    i = np.arange(n)
    tri = np.stack([i, i + 1, i + 2], 1)
    x = np.stack([i // 2, i % 2, np.zeros(n)], 1)
    xyz = np.concatenate([x, [[n // 2 + 1, 0, 0], [n // 2 + 1, 1, 0]]]).astype(np.float32)
    return mesh_of(xyz, tri[::-1] if reverse else tri)


def comb(teeth, length):
    """A spine strip with ``teeth`` strips hanging off it, every tooth numbered before the spine."""
    tris, verts = [], []
    spine = len(verts)
    for k in range(2 * teeth + 2):
        verts.append([k, 0, 0])
    for k in range(teeth):
        base = len(verts)
        a, b = spine + 2 * k, spine + 2 * k + 1
        prev = (a, b)
        for j in range(length):
            verts += [[2 * k, j + 1, 0], [2 * k + 1, j + 1, 0]]
            c, d = base + 2 * j, base + 2 * j + 1
            tris += [[prev[0], prev[1], c], [prev[1], d, c]]
            prev = (c, d)
    tris += [[spine + k, spine + k + 1, spine + k + 2] for k in range(2 * teeth)]
    return mesh_of(verts, tris)


def edge_fan(n):
    """n triangles on the single edge (0, 1)."""
    a = np.linspace(0, 2 * np.pi, n, endpoint=False)
    xyz = np.concatenate([[[0, 0, 0], [0, 0, 1]], np.stack([np.cos(a), np.sin(a), np.full(n, 0.5)], 1)])
    return mesh_of(xyz, [[0, 1, k + 2] for k in range(n)])


def isolated(n, seed=0):
    """n triangles sharing no edge."""
    rng = np.random.default_rng(seed)
    xyz = rng.random((3 * n, 3)).astype(np.float32)
    return mesh_of(xyz, np.arange(3 * n).reshape(n, 3))


def check_areas(mesh, clusters, n, area):
    """The fixed-point areas against math.fsum of the cluster's triangle areas."""
    v = np.asarray(mesh.vertices, np.float32).reshape(-1, 3)
    t = np.asarray(mesh.triangles, np.int64).reshape(-1, 3)
    if len(t) == 0:
        return
    a = CO.triangle_areas(v, t)
    s = CO.area_scale(a)
    order = np.argsort(clusters, kind="stable")
    bounds = np.searchsorted(clusters[order], np.arange(len(n) + 1))
    for c in range(len(n)):
        exact = math.fsum(a[order[bounds[c]:bounds[c + 1]]])
        tol = n[c] / (2 * s) + math.ulp(exact) + math.ulp(area[c])
        assert abs(area[c] - exact) <= tol, (c, area[c], exact, tol)


def compare(got, mesh, what=""):
    """A device triple against the oracle, bit for bit."""
    want = CO.cluster_connected_triangles(mesh)
    names = ("triangle_clusters", "cluster_n_triangles", "cluster_area")
    for g, w, name in zip(got, want, names):
        g = np.ascontiguousarray(g)
        assert g.dtype == w.dtype and g.shape == w.shape, f"{what}: {name} {g.dtype}{g.shape} != {w.dtype}{w.shape}"
        if g.tobytes() != w.tobytes():
            bad = int((g != w).sum())
            raise AssertionError(f"{what}: {name}: {bad} of {len(w)} differ")
    return want
