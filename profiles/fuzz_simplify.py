"""Randomised check of mesh simplification (simplify_mesh) against the oracle with the bounds of
tests/simplify_cases.py (counts, vertex order, rows, triangles and integral colours exact; positions and normals
within the fixed-point bounds; per-cluster branch of the quadric placement): random lattice meshes from the fuzz
lattices of profiles/fuzz_mesh.py, random triangle soups with repeated / rotated / reversed triangles and
non-integral colours, voxel sizes from below the vertex spacing to beyond the extent, both contractions; every
device result is also run twice.  Clusters whose branch sits on the determinant threshold or whose minimiser sits on
a cell face are counted as excluded.
    python profiles/fuzz_simplify.py [meshes] [seed]        (one JSON line, exit 1 on any mismatch)"""
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import image_to_pointcloud_b200 as m  # noqa: E402
from oracle import d2pc_mesh_oracle as MO  # noqa: E402  (checker only)
from profiles.fuzz_mesh import lattice  # noqa: E402
from tests.simplify_cases import compare, soup  # noqa: E402


def main(argv=None):
    argv = list(sys.argv if argv is None else argv)
    n_ex = int(argv[1]) if len(argv) > 1 else 300
    seed = int(argv[2]) if len(argv) > 2 else 2026
    rng = np.random.default_rng(seed)
    t0 = time.time()
    tot = {"meshes": 0, "vertices": 0, "triangles": 0, "clusters": 0, "quadric_clusters": 0,
           "excluded_clusters": 0, "mismatches": 0, "not_repeatable": 0}
    bad = []
    sides = [2, 3, 17, 64, 128, 129, 255, 300]
    for it in range(n_ex):
        if rng.random() < 0.6:
            R, Cc = int(rng.choice(sides)), int(rng.choice(sides))
            xyz, rgb, kind = lattice(rng, R, Cc)
            mesh = MO.grid_mesh(xyz, rgb, (R, Cc), max_angle=float(rng.choice([85.0, 89.0, 90.0])),
                                compute_normals=bool(rng.random() < 0.7),
                                keep=(rng.random(R * Cc) < 0.9) if rng.random() < 0.5 else None)
            info = dict(it=it, lattice=[R, Cc], kind=kind)
        else:
            mesh = soup(rng, int(rng.integers(1, 5000)), int(rng.integers(0, 10000)), normals=bool(rng.random() < 0.5),
                        integral=bool(rng.random() < 0.7))
            info = dict(it=it, soup=len(mesh.vertices))
        if len(mesh.vertices) == 0:
            continue
        ext = float(np.ptp(mesh.vertices.astype(np.float64), axis=0).max()) or 1.0
        vs = float(ext * 10.0 ** rng.uniform(-5, 1))
        if vs < ext / 2 ** 20:
            vs = ext / 2 ** 20
        contraction = str(rng.choice(["average", "quadric"]))
        info.update(vs=vs, contraction=contraction)
        tot["meshes"] += 1
        tot["vertices"] += len(mesh.vertices)
        tot["triangles"] += len(mesh.triangles)
        try:
            got = m.simplify_mesh(mesh, vs, contraction=contraction)
            st = compare(got, mesh, vs, contraction, str(info))
            tot["clusters"] += st["clusters"]
            tot["quadric_clusters"] += st["quadric"]
            tot["excluded_clusters"] += st["excluded"]
        except AssertionError as e:
            tot["mismatches"] += 1
            bad.append(dict(info, error=str(e)[:300]))
            continue
        again = m.simplify_mesh(mesh, vs, contraction=contraction)
        if any((a is None) != (b is None) or (a is not None and a.tobytes() != b.tobytes()) for a, b in zip(got, again)):
            tot["not_repeatable"] += 1
            bad.append(dict(info, error="not repeatable"))
    tot["seconds"] = round(time.time() - t0, 1)
    print(json.dumps({"seed": seed, "simplify": tot, "first_bad": bad[:6]}))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
