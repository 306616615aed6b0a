"""Randomised check of the point normals (estimate_normals) against the oracle: random clouds (uniform, clusters,
planes, lines, duplicates, lattices, outliers; 1 - 60 000 points), random knn and radius, and the stage's own clouds.
Covariances must be bit-exact; normals within 1e-9 rad of the oracle's where the relative eigengap is >= 1e-6, facing
the camera, and identical on a second run.   python profiles/fuzz_normals.py [examples] [seed]   (one JSON line)"""
import json
import os
import sys
import time
import warnings

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import image_to_pointcloud_b200 as m  # noqa: E402
from oracle import d2pc_normals_oracle as N  # noqa: E402  (checker only)
from oracle import d2pc_oracle as O  # noqa: E402
from profiles.fuzz_rows import KINDS, cloud  # noqa: E402
from tests import cases  # noqa: E402


def check(p, knn, radius, cam):
    """-> dict of failure counts for one cloud"""
    want_n, want_c = N.estimate_normals(p, knn=knn, radius=radius, orient_towards=cam, return_covariances=True)
    got_n, got_c = m.estimate_normals(p, knn=knn, radius=radius, orient_towards=cam, return_covariances=True)
    gc = np.ascontiguousarray(got_c[:, [0, 0, 0, 1, 1, 2], [0, 1, 2, 1, 2, 2]])
    res = {"cov_rows_differ": int((gc.view(np.uint64) != want_c.view(np.uint64)).any(1).sum())}
    w = np.linalg.eigvalsh(got_c) if len(p) else np.zeros((0, 3))
    with np.errstate(all="ignore"):
        sep = (w[:, 1] - w[:, 0]) / w[:, 2] >= 1e-6
    ang = np.arctan2(np.linalg.norm(np.cross(got_n, want_n), axis=1), np.abs((got_n * want_n).sum(1)))
    res["angle_over_1e-9"] = int((ang[sep] > 1e-9).sum())
    res["max_angle_separated"] = float(ang[sep].max(initial=0.0))
    if cam is not None:
        res["facing_away"] = int(((got_n * (np.asarray(cam) - p.astype(np.float64))).sum(1) < 0).sum())
    again = m.estimate_normals(p, knn=knn, radius=radius, orient_towards=cam)
    res["not_repeatable"] = int(again.tobytes() != got_n.tobytes())
    return res


def main(argv=None):
    argv = list(sys.argv if argv is None else argv)
    n_ex = int(argv[1]) if len(argv) > 1 else 200
    seed = int(argv[2]) if len(argv) > 2 else 2026
    rng = np.random.default_rng(seed)
    t0 = time.time()
    tot = {"examples": 0, "points": 0, "radius_examples": 0, "stage_clouds": 0, "cov_mismatches": 0,
           "cov_rows_differ": 0, "angle_over_1e-9": 0, "facing_away": 0, "not_repeatable": 0, "max_angle_separated": 0.0}
    bad = []

    def add(res, info):
        tot["examples"] += 1
        tot["points"] += info["n"]
        tot["cov_mismatches"] += res["cov_rows_differ"] > 0
        for k in ("cov_rows_differ", "angle_over_1e-9", "facing_away", "not_repeatable"):
            tot[k] += res.get(k, 0)
        tot["max_angle_separated"] = max(tot["max_angle_separated"], res["max_angle_separated"])
        if res["cov_rows_differ"] or res["angle_over_1e-9"] or res.get("facing_away") or res["not_repeatable"]:
            bad.append(dict(info, **res))

    for it in range(n_ex):
        n = int(rng.choice([1, 2, 3, 5, 29, 30, 31, 100, 1000, 5000, 20000, 60000]))
        kind = KINDS[int(rng.integers(len(KINDS)))]
        p = cloud(rng, n, kind)
        knn = int(rng.choice([1, 2, 3, 5, 10, 20, 30, 30, 30, 31, 32, 33, 48, 64]))
        radius = None
        if rng.random() < 0.3:
            ext = float(np.ptp(p, axis=0).max()) if n > 1 else 1.0
            radius = float(max(ext, 1e-6) * 10.0 ** rng.uniform(-3, -0.5))
            tot["radius_examples"] += 1
        cam = None if rng.random() < 0.2 else tuple(float(v) for v in rng.standard_normal(3) * 5)
        add(check(p, knn, radius, cam), dict(it=it, n=n, kind=kind, knn=knn, radius=radius))
    for it, (H, W, kind, dens) in enumerate([(120, 160, "uniform", "high"), (240, 320, "scene", "high"),
                                             (240, 320, "scene", "medium"), (96, 160, "ties", "high"),
                                             (180, 240, "ties", "medium"), (200, 300, "uniform", "medium")]):
        img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            p, _ = O.depth_to_point_cloud(img, cases.make_depth(H, W, 100 + it, kind), density=dens,
                                          invert=bool(it % 2))
        for knn, radius in ((30, None), (int(rng.integers(1, 65)), None), (30, 0.05)):
            tot["stage_clouds"] += 1
            add(check(p, knn, radius, (0.0, 0.0, 0.0)), dict(stage=f"{H}x{W} {kind} {dens}", n=len(p), knn=knn,
                                                             radius=radius))
    tot["seconds"] = round(time.time() - t0, 1)
    print(json.dumps({"seed": seed, "normals": tot, "first_bad": bad[:6]}))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
