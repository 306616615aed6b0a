"""Randomised check of mesh components (cluster_connected_triangles, remove_small_components) against the oracle,
bit for bit: random lattice meshes from the fuzz lattices of profiles/fuzz_mesh.py (some with a keep mask, some
simplified, some with vertices and triangles shuffled) and random triangle soups with non-manifold, degenerate and
repeated triangles; every device result is also run twice.
    python profiles/fuzz_components.py [meshes] [seed]        (one JSON line, exit 1 on any mismatch)"""
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import image_to_pointcloud_b200 as m  # noqa: E402
from oracle import d2pc_components_oracle as CO  # noqa: E402  (checker only)
from oracle import d2pc_mesh_oracle as MO  # noqa: E402
from oracle import d2pc_simplify_oracle as SO  # noqa: E402
from profiles.fuzz_mesh import lattice  # noqa: E402
from tests.components_cases import compare, shuffled, soup  # noqa: E402


def same(a, b):
    return all((x is None) == (y is None) and (x is None or x.tobytes() == y.tobytes()) for x, y in zip(a, b))


def main(argv=None):
    argv = list(sys.argv if argv is None else argv)
    n_ex = int(argv[1]) if len(argv) > 1 else 300
    seed = int(argv[2]) if len(argv) > 2 else 2026
    rng = np.random.default_rng(seed)
    t0 = time.time()
    tot = {"meshes": 0, "triangles": 0, "clusters": 0, "removed_triangles": 0, "mismatches": 0, "not_repeatable": 0}
    bad = []
    sides = [2, 3, 17, 64, 128, 129, 255, 300]
    for it in range(n_ex):
        if rng.random() < 0.6:
            R, Cc = int(rng.choice(sides)), int(rng.choice(sides))
            xyz, rgb, kind = lattice(rng, R, Cc)
            mesh = MO.grid_mesh(xyz, rgb, (R, Cc), max_angle=float(rng.choice([60.0, 85.0, 90.0])),
                                compute_normals=bool(rng.random() < 0.7),
                                keep=(rng.random(R * Cc) < 0.9) if rng.random() < 0.5 else None)
            info = dict(it=it, lattice=[R, Cc], kind=kind)
            r = rng.random()
            if r < 0.2 and len(mesh.vertices):
                mesh = SO.simplify_mesh(mesh, float(rng.choice([0.005, 0.02])))
                info["simplified"] = True
            elif r < 0.4:
                mesh = shuffled(mesh, rng)
                info["shuffled"] = True
        else:
            V = int(rng.integers(1, 5000))
            mesh = soup(rng, V, int(rng.integers(0, 3 * V)), normals=bool(rng.random() < 0.5))
            info = dict(it=it, soup=V)
        n_min = int(rng.choice([1, 2, 10, 100]))
        info["min_triangles"] = n_min
        tot["meshes"] += 1
        tot["triangles"] += len(mesh.triangles)
        try:
            got = m.cluster_connected_triangles(mesh)
            want = compare(got, mesh, str(info))
            tot["clusters"] += len(want[1])
            clean = m.remove_small_components(mesh, min_triangles=n_min)
            ref = CO.remove_small_components(mesh, min_triangles=n_min)
            assert same(clean, ref), f"{info}: remove_small_components"
            tot["removed_triangles"] += len(mesh.triangles) - len(clean.triangles)
        except AssertionError as e:
            tot["mismatches"] += 1
            bad.append(dict(info, error=str(e)[:300]))
            continue
        if not (same(got, m.cluster_connected_triangles(mesh)) and
                same(clean, m.remove_small_components(mesh, min_triangles=n_min))):
            tot["not_repeatable"] += 1
            bad.append(dict(info, error="not repeatable"))
    tot["seconds"] = round(time.time() - t0, 1)
    print(json.dumps({"seed": seed, "components": tot, "first_bad": bad[:6]}))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
