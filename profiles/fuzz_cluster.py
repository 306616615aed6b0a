"""Randomised check of density clustering (cluster_dbscan, remove_small_clusters, remove_radius_outlier) against the
oracle, bit for bit: random clouds (uniform, blobs, lines, planes, duplicates, lattices, a clipped-style clump, and
mixtures) of 1 to 20 000 points at random scales and offsets, random eps, min_points 0..40, min_size and nb_points.
Every device result is also run twice.
    python profiles/fuzz_cluster.py [clouds] [seed] [out.json]        (one JSON line, exit 1 on any mismatch)"""
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import image_to_pointcloud_b200 as m  # noqa: E402
from oracle import d2pc_cluster_oracle as CL  # noqa: E402  (checker only)


def make(rng):
    n = int(rng.choice([1, 2, 7, 100, 1000, 5000, 20000]))
    kind = rng.integers(0, 8)
    if kind == 0:
        p = rng.random((n, 3))
    elif kind == 1:
        c = rng.random((int(rng.integers(1, 20)), 3))
        p = c[rng.integers(0, len(c), n)] + rng.normal(0, rng.choice([0.001, 0.01, 0.05]), (n, 3))
    elif kind == 2:
        t = rng.random(n)
        p = np.stack([t, np.sin(7 * t), 0.2 * np.round(rng.random(n) * 3)], 1)
    elif kind == 3:
        p = rng.random((n, 3))
        p[:, int(rng.integers(0, 3))] = np.round(p[:, 0] * 4) / 4
    elif kind == 4:
        p = np.repeat(rng.random((max(1, n // 16), 3)), 16, axis=0)[:n]
    elif kind == 5:
        k = int(round(n ** (1 / 3))) + 1
        g = np.arange(k) / k
        p = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)[:n]
    elif kind == 6:
        p = rng.random((n, 3))
        p[: n // 10] = 0.3 + rng.integers(0, 5, (n // 10, 3)) * 1e-7
    else:
        p = np.concatenate([rng.random((n // 2, 3)), rng.normal(0.5, 0.02, (n - n // 2, 3))])
    p = p * rng.choice([1e-3, 1.0, 50.0]) + rng.choice([0.0, -7.0, 1e3])
    p = p[rng.permutation(len(p))].astype(np.float32)
    ext = float((p.max(0) - p.min(0)).max()) if len(p) else 1.0
    eps = max(ext, 1e-3) * float(rng.choice([0.002, 0.01, 0.03, 0.06]))
    return p, eps


def main():
    count = int(sys.argv[1]) if len(sys.argv) > 1 else 300
    seed = int(sys.argv[2]) if len(sys.argv) > 2 else 0
    out_path = sys.argv[3] if len(sys.argv) > 3 else None
    rng = np.random.default_rng(seed)
    bad, repeat_bad, t0 = [], 0, time.time()
    for it in range(count):
        p, eps = make(rng)
        if not CL.grid_fits(p, eps):
            continue
        mp = int(rng.integers(0, 41))
        ms = int(rng.integers(1, 50))
        nb = int(rng.integers(1, 30))
        rgb = (rng.random(p.shape) * 255).astype(np.float32)
        want = CL.cluster_dbscan(p, eps, mp)
        kidx, _, _ = CL.remove_small_clusters(p, eps, mp, ms)
        ridx = CL.remove_radius_outlier(p, nb, eps)
        res = []
        for _ in range(2):
            res.append((m.cluster_dbscan(p, eps, mp), m.remove_small_clusters(p, rgb, eps=eps, min_points=mp, min_size=ms),
                        m.remove_radius_outlier(p, rgb, nb_points=nb, radius=eps)))
        g, (gp, gc, gi), (rp, rc, ri) = res[0]
        ok = (np.array_equal(g, want) and np.array_equal(gi, kidx) and gp.tobytes() == p[kidx].tobytes()
              and gc.tobytes() == rgb[kidx].tobytes() and np.array_equal(ri, ridx) and rp.tobytes() == p[ridx].tobytes())
        if not ok:
            bad.append({"it": it, "n": len(p), "eps": eps, "min_points": mp})
        a, b = res
        same = a[0].tobytes() == b[0].tobytes() and all(x.tobytes() == y.tobytes() for x, y in zip(a[1] + a[2], b[1] + b[2]))
        repeat_bad += 0 if same else 1
    out = {"clouds": count, "seed": seed, "mismatches": len(bad), "repeat_mismatches": repeat_bad, "first_bad": bad[:5],
           "seconds": round(time.time() - t0, 1)}
    line = json.dumps(out)
    print(line)
    if out_path:
        os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
        open(out_path, "w").write(line + "\n")
    sys.exit(1 if bad or repeat_bad else 0)


if __name__ == "__main__":
    main()
