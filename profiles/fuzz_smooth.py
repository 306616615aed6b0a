"""Randomised check of mesh smoothing (filter_smooth_simple / _laplacian / _taubin) and compute_vertex_normals
against the oracle, bit for bit: random lattice meshes from the fuzz lattices of profiles/fuzz_mesh.py (some with a
keep mask, some simplified, some shuffled), random triangle soups with non-manifold, degenerate and repeated
triangles, stars whose hub takes every segment-sort path, and meshes with isolated vertices or no triangles; random
method, iterations, scope, lambda and mu.  Every device result is also run twice.
    python profiles/fuzz_smooth.py [meshes] [seed]        (one JSON line, exit 1 on any mismatch)"""
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import image_to_pointcloud_b200 as m  # noqa: E402
from oracle import d2pc_mesh_oracle as MO  # noqa: E402
from oracle import d2pc_simplify_oracle as SO  # noqa: E402
from oracle import d2pc_smooth_oracle as SMO  # noqa: E402  (checker only)
from profiles.fuzz_mesh import lattice  # noqa: E402
from tests.components_cases import mesh_of, shuffled, soup  # noqa: E402

FUNCS = {"simple": m.filter_smooth_simple, "laplacian": m.filter_smooth_laplacian, "taubin": m.filter_smooth_taubin}


def same(a, b):
    return all((x is None) == (y is None) and (x is None or np.ascontiguousarray(x).tobytes() == y.tobytes())
               for x, y in zip(a, b))


def star(rng, n):
    a = np.sort(rng.random(n)) * 2 * np.pi
    xyz = np.concatenate([[[0, 0, 0.3]], np.stack([np.cos(a), np.sin(a), 0.1 * rng.random(n)], 1)])
    k = np.arange(n)
    return mesh_of(xyz, np.stack([np.zeros(n, np.int64), k + 1, (k + 1) % n + 1], 1), bool(rng.random() < 0.5),
                   int(rng.integers(1 << 30)))


def make(rng, it):
    r = rng.random()
    if r < 0.5:
        sides = [2, 3, 17, 64, 128, 129, 255]
        R, Cc = int(rng.choice(sides)), int(rng.choice(sides))
        xyz, rgb, kind = lattice(rng, R, Cc)
        mesh = MO.grid_mesh(xyz, rgb, (R, Cc), max_angle=float(rng.choice([60.0, 85.0, 90.0])),
                            compute_normals=bool(rng.random() < 0.7),
                            keep=(rng.random(R * Cc) < 0.9) if rng.random() < 0.5 else None)
        info = dict(it=it, lattice=[R, Cc], kind=kind)
        q = rng.random()
        if q < 0.2 and len(mesh.vertices):
            mesh = SO.simplify_mesh(mesh, float(rng.choice([0.005, 0.02])))
            info["simplified"] = True
        elif q < 0.4:
            mesh = shuffled(mesh, rng)
            info["shuffled"] = True
        return mesh, info
    if r < 0.8:
        V = int(rng.integers(1, 3000))
        return soup(rng, V, int(rng.integers(0, 3 * V)), normals=bool(rng.random() < 0.5)), dict(it=it, soup=V)
    if r < 0.9:
        n = int(rng.choice([3, 31, 32, 33, 500, 4095, 4096, 4097, 9000]))
        return star(rng, n), dict(it=it, star=n)
    V = int(rng.integers(0, 200))
    T = int(rng.integers(0, 2)) * int(rng.integers(1, max(V // 3, 1) + 1)) if V else 0
    tri = rng.integers(0, max(V, 1), (T, 3)) if V else np.zeros((0, 3))
    return mesh_of(rng.random((V, 3)), tri, bool(rng.random() < 0.5), int(rng.integers(1 << 30))), dict(it=it, sparse=V)


def main(argv=None):
    argv = list(sys.argv if argv is None else argv)
    n_ex = int(argv[1]) if len(argv) > 1 else 300
    seed = int(argv[2]) if len(argv) > 2 else 2026
    rng = np.random.default_rng(seed)
    t0 = time.time()
    tot = {"meshes": 0, "vertices": 0, "triangles": 0, "passes": 0, "mismatches": 0, "not_repeatable": 0}
    bad = []
    for it in range(n_ex):
        mesh, info = make(rng, it)
        method = str(rng.choice(SMO.METHODS))
        n = int(rng.choice([0, 1, 2, 3, 5, 10]))
        scope = str(rng.choice(list(SMO.SCOPES)))
        lam, mu = (0.5, -0.53) if rng.random() < 0.5 else (float(rng.uniform(-1, 1)), float(rng.uniform(-1, 1)))
        info.update(method=method, iterations=n, scope=scope, lam=lam, mu=mu)
        kw = dict(scope=scope)
        if method != "simple":
            kw["lambda_filter"] = lam
        if method == "taubin":
            kw["mu"] = mu
        tot["meshes"] += 1
        tot["vertices"] += len(mesh.vertices)
        tot["triangles"] += len(mesh.triangles)
        tot["passes"] += n * (2 if method == "taubin" else 1)
        try:
            got = FUNCS[method](mesh, n, **kw)
            want = SMO.filter_smooth(mesh, method, n, lam, mu, scope)
            assert same(got, want), f"{info}: smoothing"
            nrm = m.compute_vertex_normals(mesh)
            assert same(nrm, SMO.compute_vertex_normals(mesh)), f"{info}: normals"
        except AssertionError as e:
            tot["mismatches"] += 1
            bad.append(dict(info, error=str(e)[:300]))
            continue
        if not (same(got, [None if x is None else np.ascontiguousarray(x) for x in FUNCS[method](mesh, n, **kw)])
                and same(nrm, [None if x is None else np.ascontiguousarray(x) for x in m.compute_vertex_normals(mesh)])):
            tot["not_repeatable"] += 1
            bad.append(dict(info, error="not repeatable"))
    tot["seconds"] = round(time.time() - t0, 1)
    print(json.dumps({"seed": seed, "smooth": tot, "first_bad": bad[:6]}))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
