"""TEST INFRASTRUCTURE ONLY -- CPU oracle for mesh smoothing and the vertex normals of any mesh (DESIGN row m4).

SPEC FROZEN HERE, NO REFERENCE CODE: the reference smooths its meshes through Open3D's Poisson reconstruction
(backend/app.py:271-308).  This restates Open3D's ``TriangleMesh::FilterSmoothSimple``, ``FilterSmoothLaplacian``,
``FilterSmoothTaubin`` and ``ComputeAdjacencyList`` (geometry/TriangleMesh.cpp); Open3D is not installed in the build
container, so parity is UNPINNED.  The product package never imports this module.

Input: a mesh in the ``TriangleMesh`` layout (vertices f32 [V, 3], colors f32 [V, 3] (0..255), triangles i32 [T, 3],
vertex_normals f64 [V, 3] or None, vertex_rows i64 [V]).

  errors      a triangle id < 0 or >= V; a non-finite vertex coordinate, or a non-finite colour / normal when the
              scope filters it (ValueError)
  adjacency   Open3D's ComputeAdjacencyList: triangle (a, b, c) adds b, c to adj[a], a, c to adj[b], a, b to adj[c],
              as sets ((a, a, b) puts a in adj[a]); DEPARTURE: neighbours are visited in ascending vertex id (Open3D
              iterates an unordered_set)
  state       float64 (the float32 input widened); every pass reads the previous state and writes a new one (Jacobi);
              rounded to float32 once at the end (normals stay float64)
  scope       "all", "vertex", "normal", "color" (Open3D's FilterScope); normals only when the mesh has them; the
              other fields are copied; filtered normals are not renormalised
  simple      p' = (p + sum_nb p_nb) / (1 + |adj|), the sum left to right in neighbour order from zero
  laplacian   per neighbour d = sqrt((dx*dx + dy*dy) + dz*dz) of diff = p - p_nb, w = 1 / (d + 1e-12), W += w,
              S += w * p_nb (left to right from zero); p' = p + lambda * (S / W - p) per component.  Colours and
              normals take the same weights (from positions).  DEPARTURE: a vertex without neighbours stays as it is
              (Open3D computes 0 / 0)
  taubin      every iteration one laplacian pass with lambda, then one with mu (Open3D: 0.5, -0.53)
  iterations  0 returns a copy; triangles and vertex rows never change
  normals     ``compute_vertex_normals``: m1's rule (d2pc_mesh_oracle._finish, which this module calls): the
              unnormalised (p1 - p0) x (p2 - p0) of every triangle from the float32 vertices as float64, summed per
              vertex in ascending triangle order once per corner, then v / sqrt(v.v), (0, 0, 1) for a zero sum

Two restatements: the vectorised one below (the k-th neighbour of every vertex at once, k = 0, 1, ..., so every sum
runs left to right) and ``filter_smooth_loop`` / ``compute_vertex_normals_loop`` (Open3D's per-vertex loops over
Python floats, the sets sorted), which the CPU tests check against each other.
"""
from __future__ import annotations

import math

import numpy as np

from .d2pc_components_oracle import check_mesh
from .d2pc_mesh_oracle import Mesh, _finish
from .d2pc_oracle import F64

METHODS = ("simple", "laplacian", "taubin")
SCOPES = {"all": ("vertex", "normal", "color"), "vertex": ("vertex",), "normal": ("normal",), "color": ("color",)}
EPS = 1e-12


def _check(mesh, scope):
    if scope not in SCOPES:
        raise ValueError(f"scope must be one of {tuple(SCOPES)}")
    v, t = check_mesh(mesh)
    fields = SCOPES[scope]
    c = np.asarray(mesh.colors, np.float32).reshape(-1, 3)
    n = None if mesh.vertex_normals is None else np.asarray(mesh.vertex_normals, F64).reshape(-1, 3)
    if "color" in fields and not np.isfinite(c).all():
        raise ValueError("the mesh has a non-finite colour")
    if "normal" in fields and n is not None and not np.isfinite(n).all():
        raise ValueError("the mesh has a non-finite normal")
    return v, c, n, t


def adjacency(V: int, t: np.ndarray):
    """(offsets int64 [V + 1], neighbours int64 [E]): every vertex's neighbour set in ascending order."""
    t = np.asarray(t, np.int64).reshape(-1, 3)
    a, b = t.reshape(-1), np.roll(t, -1, axis=1).reshape(-1)
    keys = np.unique((np.minimum(a, b) << 32) | np.maximum(a, b))
    lo, hi = keys >> 32, keys & 0xFFFFFFFF
    off_diag = lo != hi
    src = np.concatenate([lo, hi[off_diag]])
    dst = np.concatenate([hi, lo[off_diag]])
    order = np.lexsort((dst, src))
    src, dst = src[order], dst[order]
    off = np.zeros(V + 1, np.int64)
    np.cumsum(np.bincount(src, minlength=V), out=off[1:])
    return off, dst


def _slots(off: np.ndarray):
    """[(vertices, entries)] of slot k = 0, 1, ...: the k-th entry of every segment that has one."""
    deg = np.diff(off)
    V = len(deg)
    src = np.repeat(np.arange(V), deg)
    rank = np.arange(len(src)) - off[src]
    order = np.argsort(rank, kind="stable")
    bounds = np.searchsorted(rank[order], np.arange(int(deg.max()) + 2 if V and len(src) else 1))
    return [(src[order[bounds[k]:bounds[k + 1]]], order[bounds[k]:bounds[k + 1]]) for k in range(len(bounds) - 1)]


def _pass(state, filt, off, nbr, slots, method, lam):
    """One Jacobi pass: state = [positions, colours, normals or None] (float64), filt = which of them to filter."""
    deg = np.diff(off)
    out = list(state)
    if method == "simple":
        for f in range(3):
            if not filt[f]:
                continue
            x = state[f]
            s = np.zeros_like(x)
            for vs, ent in slots:
                s[vs] = s[vs] + x[nbr[ent]]
            out[f] = (x + s) / (1 + deg)[:, None]
        return out
    p = state[0]
    W = np.zeros(len(p))
    S = [np.zeros_like(x) if filt[f] else None for f, x in enumerate(state)]
    for vs, ent in slots:
        nb = nbr[ent]
        d = p[vs] - p[nb]
        w = 1.0 / (np.sqrt((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]) + EPS)
        W[vs] = W[vs] + w
        for f in range(3):
            if filt[f]:
                S[f][vs] = S[f][vs] + w[:, None] * state[f][nb]
    has = deg > 0
    for f in range(3):
        if filt[f]:
            x = state[f].copy()
            x[has] = state[f][has] + lam * (S[f][has] / W[has][:, None] - state[f][has])
            out[f] = x
    return out


def _passes(method, iterations, lam, mu):
    if method not in METHODS:
        raise ValueError(f"method must be one of {METHODS}")
    n = int(iterations)
    if n != iterations or n < 0:
        raise ValueError("number_of_iterations must be an integer >= 0")
    if not (math.isfinite(lam) and math.isfinite(mu)):
        raise ValueError("lambda_filter and mu must be finite")
    if method == "taubin":
        return [("laplacian", lam), ("laplacian", mu)] * n
    return [(method, lam)] * n


def _result(mesh, v, c, n, t, state):
    return Mesh(state[0].astype(np.float32), state[1].astype(np.float32), t.astype(np.int32),
                state[2] if n is not None else None, np.asarray(mesh.vertex_rows, np.int64).reshape(-1).copy())


def filter_smooth(mesh, method: str, number_of_iterations: int = 1, lambda_filter: float = 0.5, mu: float = -0.53,
                  scope: str = "all") -> Mesh:
    """Vectorised restatement of the spec (module docstring)."""
    passes = _passes(method, number_of_iterations, lambda_filter, mu)
    v, c, n, t = _check(mesh, scope)
    fields = SCOPES[scope]
    filt = ("vertex" in fields, "color" in fields, "normal" in fields and n is not None)
    state = [v.astype(F64), c.astype(F64), None if n is None else n.copy()]
    off, nbr = adjacency(len(v), t)
    slots = _slots(off)
    for m, lam in passes:
        state = _pass(state, filt, off, nbr, slots, m, lam)
    return _result(mesh, v, c, n, t, state)


def filter_smooth_simple(mesh, number_of_iterations=1, scope="all") -> Mesh:
    return filter_smooth(mesh, "simple", number_of_iterations, scope=scope)


def filter_smooth_laplacian(mesh, number_of_iterations=1, lambda_filter=0.5, scope="all") -> Mesh:
    return filter_smooth(mesh, "laplacian", number_of_iterations, lambda_filter, scope=scope)


def filter_smooth_taubin(mesh, number_of_iterations=1, lambda_filter=0.5, mu=-0.53, scope="all") -> Mesh:
    return filter_smooth(mesh, "taubin", number_of_iterations, lambda_filter, mu, scope)


def compute_vertex_normals(mesh) -> Mesh:
    """The mesh with m1's vertex normals (``d2pc_mesh_oracle._finish`` on the mesh's own triangles)."""
    v, t = check_mesh(mesh)
    nrm = _finish(v, np.zeros_like(v), len(v), np.ones(len(v), bool), t, False, True).vertex_normals
    return Mesh(v.copy(), np.asarray(mesh.colors, np.float32).reshape(-1, 3).copy(), t.astype(np.int32), nrm,
                np.asarray(mesh.vertex_rows, np.int64).reshape(-1).copy())


# --------------------------------------------------------------------------------------------
# the literal restatement: Open3D's loops over Python floats
# --------------------------------------------------------------------------------------------
def adjacency_loop(V: int, t) -> list:
    adj = [set() for _ in range(V)]
    for a, b, c in (tuple(int(x) for x in row) for row in np.asarray(t).reshape(-1, 3)):
        adj[a].update((b, c))
        adj[b].update((a, c))
        adj[c].update((a, b))
    return [sorted(s) for s in adj]


def _pass_loop(state, filt, adj, method, lam):
    out = [None if x is None else [list(r) for r in x] for x in state]
    for i, nbs in enumerate(adj):
        if method == "simple":
            for f in range(3):
                if filt[f]:
                    s = [0.0, 0.0, 0.0]
                    for j in nbs:
                        for k in range(3):
                            s[k] += state[f][j][k]
                    out[f][i] = [(state[f][i][k] + s[k]) / (1 + len(nbs)) for k in range(3)]
            continue
        if not nbs:
            continue
        p = state[0][i]
        tw = 0.0
        s = [[0.0, 0.0, 0.0] for _ in range(3)]
        for j in nbs:
            q = state[0][j]
            dx, dy, dz = p[0] - q[0], p[1] - q[1], p[2] - q[2]
            w = 1.0 / (math.sqrt((dx * dx + dy * dy) + dz * dz) + EPS)
            tw += w
            for f in range(3):
                if filt[f]:
                    for k in range(3):
                        s[f][k] += w * state[f][j][k]
        for f in range(3):
            if filt[f]:
                out[f][i] = [state[f][i][k] + lam * (s[f][k] / tw - state[f][i][k]) for k in range(3)]
    return out


def filter_smooth_loop(mesh, method: str, number_of_iterations: int = 1, lambda_filter: float = 0.5,
                       mu: float = -0.53, scope: str = "all") -> Mesh:
    passes = _passes(method, number_of_iterations, lambda_filter, mu)
    v, c, n, t = _check(mesh, scope)
    fields = SCOPES[scope]
    filt = ("vertex" in fields, "color" in fields, "normal" in fields and n is not None)
    state = [[[float(x) for x in r] for r in a] if a is not None else None for a in (v, c, n)]
    adj = adjacency_loop(len(v), t)
    for m, lam in passes:
        state = _pass_loop(state, filt, adj, m, lam)
    arr = [np.array(x, F64).reshape(-1, 3) if x is not None else None for x in state]
    return _result(mesh, v, c, n, t, arr)


def compute_vertex_normals_loop(mesh) -> Mesh:
    """Open3D's ComputeVertexNormals: every triangle's normal added to its three corners in triangle order."""
    v, t = check_mesh(mesh)
    P = [[float(x) for x in r] for r in v]
    acc = [[0.0, 0.0, 0.0] for _ in P]
    for a, b, c in (tuple(int(x) for x in row) for row in t):
        u = [P[b][k] - P[a][k] for k in range(3)]
        w = [P[c][k] - P[a][k] for k in range(3)]
        n = (u[1] * w[2] - u[2] * w[1], u[2] * w[0] - u[0] * w[2], u[0] * w[1] - u[1] * w[0])
        for i in (a, b, c):
            for k in range(3):
                acc[i][k] += n[k]
    out = []
    for s in acc:
        ss = (s[0] * s[0] + s[1] * s[1]) + s[2] * s[2]
        out.append([0.0, 0.0, 1.0] if ss == 0.0 else [x / math.sqrt(ss) for x in s])
    return Mesh(v.copy(), np.asarray(mesh.colors, np.float32).reshape(-1, 3).copy(), t.astype(np.int32),
                np.array(out, F64).reshape(-1, 3), np.asarray(mesh.vertex_rows, np.int64).reshape(-1).copy())
