"""Meshes and the device-against-oracle comparison for mesh simplification (row m2), shared by
tests/test_simplify_gpu.py and profiles/fuzz_simplify.py.

What must match exactly: counts, vertex order (vertex_rows), triangles, and colours when the input colours are
integral.  The rest is held to the bounds of the device's 64-bit fixed-point sums:
  average positions  2^-38 * E (E = the mesh's extent) plus one float32 ulp
  quadric positions  ||A^-1|| (||dA|| ||x|| + ||db||) from the quanta of the A and b sums, plus one float32 ulp
  normals            1e-9 rad where the sum's length is >= 1e-6 * count
  branch             the same per cluster, except where the normalised determinant lies within a relative 1e-9 (or
                     the fixed-point bound) of the threshold, or the minimiser within 1e-9 vs (or its tolerance) of a
                     cell face; those are counted as excluded
"""
from __future__ import annotations

import math

import numpy as np

from oracle import d2pc_mesh_oracle as MO
from oracle import d2pc_simplify_oracle as SO


def _pow2_at_least(x: float) -> float:
    """2^ex with x < 2^ex (frexp), 1 for x <= 0."""
    if not x > 0.0:
        return 1.0
    return math.ldexp(1.0, math.frexp(x)[1])


def compare(got, mesh, vs: float, contraction: str, what: str = "") -> dict:
    """Checks a device result against the oracle; returns counts of the checked and excluded clusters."""
    d = SO.Detail()
    want = SO.simplify_mesh(mesh, vs, contraction, detail=d)
    got = MO.Mesh(*(None if a is None else np.ascontiguousarray(a) for a in got))
    k = len(want.vertices)
    assert len(got.vertices) == k and len(got.triangles) == len(want.triangles), \
        f"{what}: counts {len(got.vertices)}/{len(got.triangles)} != {k}/{len(want.triangles)}"
    assert got.vertex_rows.dtype == np.int64 and np.array_equal(got.vertex_rows, want.vertex_rows), f"{what}: rows"
    assert got.triangles.dtype == np.int32 and np.array_equal(got.triangles, want.triangles), f"{what}: triangles"
    stats = dict(clusters=k, excluded=0, quadric=0)
    if k == 0:
        return stats
    col = np.asarray(mesh.colors, np.float32)
    if np.array_equal(col, np.round(col)):
        assert got.colors.tobytes() == want.colors.tobytes(), f"{what}: colours"
    else:
        cm = float(np.abs(col.astype(np.float64)).max())
        tol = _pow2_at_least(cm) * 2.0 ** -38 + np.spacing(np.abs(want.colors))
        assert (np.abs(got.colors.astype(np.float64) - want.colors) <= tol).all(), f"{what}: colours"
    p = np.asarray(mesh.vertices, np.float32).astype(np.float64)
    E = float(np.ptp(p, axis=0).max())
    avg_f32 = SO._exact_sums(p, d["cid"], k, 24, True).astype(np.float32)
    avg_tol = _pow2_at_least(E) * 2.0 ** -38 + np.spacing(np.abs(avg_f32)).astype(np.float64)
    gv = got.vertices.astype(np.float64)
    near_avg = (np.abs(gv - avg_f32) <= avg_tol).all(axis=1)
    if contraction == "average":
        assert near_avg.all(), f"{what}: {int((~near_avg).sum())} average positions off"
    else:
        A, b, x = d["A"], d["b"], d["x"] - d["bmin"][None, :]
        t = np.asarray(mesh.triangles, np.int64).reshape(-1, 3)
        areas = SO.triangle_quadrics(p - d["bmin"][None, :], t)[0] if len(t) else np.zeros((0, 6))
        area_sum = float(((areas[:, 0] + areas[:, 3]) + areas[:, 5]).sum()) if len(t) else 0.0
        qa = _pow2_at_least(3.0 * area_sum * (1 + 2.0 ** -19)) * 2.0 ** -61
        qb = _pow2_at_least(3.0 * area_sum * (1 + 2.0 ** -19) * math.sqrt(3) * _pow2_at_least(E)) * 2.0 ** -61
        kc = np.bincount(d["cid"][t].reshape(-1), minlength=k).astype(np.float64) if len(t) else np.zeros(k)
        eps = 2.0 ** -52
        dA = kc * (qa + eps * np.abs(A).max(axis=1))          # per entry: fixed-point quanta + float64 sums
        db = kc * (qb + eps * np.abs(b).max(axis=1))
        M = np.zeros((k, 3, 3))
        iu = np.triu_indices(3)
        M[:, iu[0], iu[1]] = A
        M[:, iu[1], iu[0]] = A
        with np.errstate(all="ignore"):
            inv_norm = 1.0 / np.abs(np.linalg.eigvalsh(M)).min(axis=1)   # ||A^-1||_2
            dx = 4.0 * inv_norm * (3.0 * dA * np.linalg.norm(x, axis=1) + math.sqrt(3.0) * db)
        xq = d["x"].astype(np.float32)
        q_tol = dx[:, None] + np.spacing(np.abs(xq)).astype(np.float64)
        near_q = (np.abs(gv - xq.astype(np.float64)) <= q_tol).all(axis=1)
        tr, det = d["trace"], d["det"]
        with np.errstate(all="ignore"):
            rel = np.abs(det / (tr * tr * tr) / SO.DET_REL - 1.0)
            # det is cubic in entries bounded by t: |d det| <= 18 dA t^2, i.e. 18 dA / t on det / t^3
            det_margin = np.maximum(1e-9, 18.0 * dA / np.maximum(tr, 1e-300) / SO.DET_REL)
            face = np.minimum(np.abs(d["x"] - d["lo"]), np.abs(d["x"] - d["hi"])).min(axis=1)
        ambiguous = (rel <= det_margin) | (face <= np.maximum(1e-9 * vs, dx))
        ok = np.where(d["quadric"], near_q, near_avg)
        bad = ~ok & ~ambiguous
        assert not bad.any(), f"{what}: {int(bad.sum())} of {k} clusters off (first {np.nonzero(bad)[0][:5]})"
        stats["excluded"] = int((~ok & ambiguous).sum())
        stats["quadric"] = int(d["quadric"].sum())
    if want.vertex_normals is not None:
        assert got.vertex_normals is not None and got.vertex_normals.dtype == np.float64
        nrm = np.asarray(mesh.vertex_normals, np.float64)
        s = np.zeros((k, 3))
        np.add.at(s, d["cid"], nrm)
        sel = np.linalg.norm(s, axis=1) >= 1e-6 * d["count"]
        g, w = got.vertex_normals[sel], want.vertex_normals[sel]
        ang = np.arctan2(np.linalg.norm(np.cross(g, w), axis=1), (g * w).sum(axis=1))
        assert (ang <= 1e-9).all() and (np.abs(np.linalg.norm(g, axis=1) - 1) <= 1e-12).all(), f"{what}: normals"
    else:
        assert got.vertex_normals is None
    return stats


def soup(rng, V, T, dup=0.2, normals=True, integral=True, spread=None):
    """A random triangle soup with repeated, rotated and reversed triangles."""
    spread = float(rng.choice([0.5, 3.0, 40.0])) if spread is None else spread
    xyz = (rng.random((V, 3)) * spread + rng.normal(0, 5, 3)).astype(np.float32)
    rgb = rng.integers(0, 256, (V, 3)).astype(np.float32) if integral else (rng.random((V, 3)) * 255).astype(np.float32)
    tri = rng.integers(0, max(V, 1), (T, 3)).astype(np.int32)
    k = int(T * dup)
    if k and T:
        src = tri[rng.integers(0, T, k)]
        src = np.stack([np.roll(r, s) for r, s in zip(src, rng.integers(0, 3, k))])
        rev = rng.random(k) < 0.3
        src[rev] = src[rev][:, ::-1]
        tri = np.concatenate([tri, src])[rng.permutation(T + k)]
    nrm = None
    if normals:
        nrm = rng.normal(size=(V, 3))
        nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    return MO.Mesh(xyz, rgb, tri, nrm, rng.permutation(10 * max(V, 1))[:V].astype(np.int64))
