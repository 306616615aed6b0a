"""Randomised check of the lattice mesh (grid_mesh) against the oracle, bit for bit: random lattice shapes (sides 1,
the tile width +-1, up to 300 x 400), random depth fields (smooth, steps, noise, constant planes, near-zero apex
points, NaN / inf rows), random keep masks and options (max_edge, max_angle, remove_unreferenced, normals), and the
stage's own lattices; every device result is also run twice.
    python profiles/fuzz_mesh.py [clouds] [seed]        (one JSON line, exit 1 on any mismatch)"""
import json
import os
import sys
import time
import warnings

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import image_to_pointcloud_b200 as m  # noqa: E402
from oracle import d2pc_mesh_oracle as MO  # noqa: E402  (checker only)
from oracle import d2pc_oracle as O  # noqa: E402
from tests import cases  # noqa: E402


def lattice(rng, R, Cc):
    kind = str(rng.choice(["smooth", "steps", "noise", "plane", "apex", "mixed"]))
    v, u = np.mgrid[0:R, 0:Cc].astype(np.float64)
    if kind == "smooth":
        z = 5 + np.sin(u / 7.0) + np.cos(v / 5.0)
    elif kind == "steps":
        z = 2 + 4 * (rng.random((R, Cc)) < 0.3) + rng.random((R, Cc)) * 0.01
    elif kind == "noise":
        z = rng.random((R, Cc)) * 20
    elif kind == "plane":
        z = np.full((R, Cc), float(rng.uniform(0.5, 10)))
    elif kind == "apex":
        z = rng.random((R, Cc)) * 10
        z[rng.random((R, Cc)) < 0.3] = 0.0
    else:
        z = np.round(rng.random((R, Cc)) * 4) * 2.5
    f = float(rng.uniform(50, 2000))
    zz = np.where(z != 0.0, z, 1e-6)
    xyz = np.stack([(u - Cc / 2) * zz / f, (v - R / 2) * zz / f, z], -1).reshape(-1, 3).astype(np.float32)
    if rng.random() < 0.5:
        bad = rng.random(R * Cc) < rng.uniform(0, 0.2)
        xyz[bad, int(rng.integers(3))] = rng.choice([np.nan, np.inf, -np.inf])
    rgb = rng.integers(0, 256, (R * Cc, 3)).astype(np.float32)
    return xyz, rgb, kind


def compare(got, want):
    return [f for f, a, b in zip(MO.Mesh._fields, got, want)
            if (a is None) != (b is None) or (a is not None and (a.shape != b.shape or a.dtype != b.dtype
                                                               or a.tobytes() != b.tobytes()))]


def main(argv=None):
    argv = list(sys.argv if argv is None else argv)
    n_ex = int(argv[1]) if len(argv) > 1 else 500
    seed = int(argv[2]) if len(argv) > 2 else 2026
    rng = np.random.default_rng(seed)
    t0 = time.time()
    tot = {"clouds": 0, "rows": 0, "triangles": 0, "stage_clouds": 0, "mismatches": 0, "not_repeatable": 0}
    bad = []

    def run(xyz, rgb, shape, kw, info):
        want = MO.grid_mesh(xyz, rgb, shape, **kw)
        got = m.grid_mesh(xyz, rgb, shape, **kw)
        again = m.grid_mesh(xyz, rgb, shape, **kw)
        diff = compare(got, want)
        rep = compare(again, got)
        tot["clouds"] += 1
        tot["rows"] += len(xyz)
        tot["triangles"] += len(want.triangles)
        tot["mismatches"] += bool(diff)
        tot["not_repeatable"] += bool(rep)
        if diff or rep:
            bad.append(dict(info, differ=diff, repeat=rep, **{k: (v if not isinstance(v, np.ndarray) else "mask")
                                                            for k, v in kw.items()}))

    sides = [1, 2, 3, 5, 17, 64, 127, 128, 129, 255, 256, 257, 300, 400]
    for it in range(n_ex):
        R, Cc = int(rng.choice(sides)), int(rng.choice(sides))
        xyz, rgb, kind = lattice(rng, R, Cc)
        kw = dict(max_angle=float(rng.choice([85.0, 90.0, 89.9, 60.0, float(rng.uniform(1, 90))])),
                  remove_unreferenced=bool(rng.random() < 0.7), compute_normals=bool(rng.random() < 0.8))
        if rng.random() < 0.4:
            kw["max_edge"] = float(10.0 ** rng.uniform(-3, 1))
        if rng.random() < 0.5:
            kw["keep"] = rng.random(R * Cc) < rng.uniform(0.3, 1.0)
        run(xyz, rgb, (R, Cc), kw, dict(it=it, shape=[R, Cc], kind=kind))
    for it, (H, W, kind, dens) in enumerate([(120, 160, "uniform", "high"), (240, 320, "scene", "high"),
                                             (241, 323, "scene", "medium"), (96, 160, "ties", "high"),
                                             (181, 243, "ties", "medium"), (200, 300, "uniform", "medium"),
                                             (518, 924, "scene", "high")]):
        img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            xyz, rgb = O.depth_to_point_cloud(img, cases.make_depth(H, W, 100 + it, kind), density=dens,
                                              invert=bool(it % 2 == 0))
        s = O.DENSITY_STEP[dens]
        shape = (-(-H // s), -(-W // s))
        for kw in (dict(), dict(max_angle=90.0, remove_unreferenced=False), dict(max_edge=0.05, max_angle=80.0)):
            tot["stage_clouds"] += 1
            run(xyz, rgb, shape, kw, dict(stage=f"{H}x{W} {kind} {dens}"))
    tot["seconds"] = round(time.time() - t0, 1)
    print(json.dumps({"seed": seed, "mesh": tot, "first_bad": bad[:6]}))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
