"""Randomised check of the voxel grid (row ax-2) against the oracle, fed straight into the kernels: random synthetic
clouds (tests/voxel_cases.py: uniform, clusters, planes, lines, duplicates, negative and far-off clouds, voxel faces,
runs across 32-row groups and 1024-row tiles, lattices), random batches of frames of different sizes sharing one table,
random densities on the same engine, fused and split inserts.  Every frame must have the oracle's voxels and
indices, bit-exact colour means and coordinate means within 2^-38 * E + ulp_f32 of the exact means; the fused insert
run twice and the split insert must give the same bits.
    python profiles/fuzz_voxel.py [batches] [seed]        (one JSON line, exit 1 on any mismatch)"""
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import image_to_pointcloud_b200 as m  # noqa: E402
from tests import voxel_cases as V  # noqa: E402  (generators and the checker; the oracle is the reference)

GEOMETRIES = [(60, 80), (240, 320), (97, 1031), (512, 512)]
SIZES = [1, 2, 3, 31, 32, 33, 100, 1023, 1024, 1025, 5000, 20000, 70000]


def main(argv=None):
    argv = list(sys.argv if argv is None else argv)
    n_batches = int(argv[1]) if len(argv) > 1 else 300
    seed = int(argv[2]) if len(argv) > 2 else 2027
    rng = np.random.default_rng(seed)
    t0 = time.time()
    engines = {}
    tot = {"batches": 0, "frames": 0, "rows": 0, "voxels": 0, "mismatches": 0, "not_repeatable": 0,
           "split_differs": 0, "worst_err_over_bound": 0.0}
    kinds = {}
    bad = []
    for it in range(n_batches):
        H, W = GEOMETRIES[int(rng.integers(len(GEOMETRIES)))]
        B = int(rng.integers(1, 6))
        if (H, W, B) not in engines:
            engines[(H, W, B)] = m.FrameEngine(H, W, batch=B)
        eng = engines[(H, W, B)]
        density = str(rng.choice(["high", "medium", "low"]))
        zr = (0.5, 9.5) if rng.random() < 0.3 else None
        cfg = eng.make_config(density=density, z_range=zr, want_bounds=True)
        N = eng.points_per_frame(cfg)
        frames = []
        for _ in range(B):
            n = min(N, int(rng.choice(SIZES + [0, N])))
            if n == 0:
                frames.append((np.zeros((0, 3), np.float32), np.zeros((0, 3), np.float32)))
                continue
            p, kind = V.random_cloud(rng, n)
            p = p[:N]
            kinds[kind] = kinds.get(kind, 0) + 1
            frames.append((p, V.colours(rng, len(p), str(rng.choice(["random", "white", "black_white"])))))
        nonempty = [p for p, _ in frames if len(p)]
        vs = V.fuzz_voxel_size(rng, nonempty[0]) if nonempty else 0.1
        # one voxel size per call: large enough for every frame's indices to stay below 2^21
        vs = max([vs] + [V.extent(p) * 2.0 ** -20 for p in nonempty])
        split = bool(rng.random() < 0.5)
        got, _ = V.run_device(eng, cfg, frames, vs, split=split)
        again, _ = V.run_device(eng, cfg, frames, vs, split=not split)
        tot["batches"] += 1
        for b, ((p, c), g, a) in enumerate(zip(frames, got, again)):
            problems, ratio = V.check_frame(*g, p, c, vs, what=f"batch {it} frame {b}")
            tot["frames"] += 1
            tot["rows"] += len(p)
            tot["voxels"] += len(g[0])
            if np.isfinite(ratio):
                tot["worst_err_over_bound"] = max(tot["worst_err_over_bound"], ratio)
            differs = V.canonical(*g) != V.canonical(*a)
            tot["mismatches"] += bool(problems)
            tot["split_differs"] += bool(differs)
            if problems or differs:
                bad.append(dict(it=it, frame=b, geometry=[H, W, B], density=density, rows=len(p), vs=vs,
                                problems=problems[:2], split_differs=bool(differs)))
        # the same call once more (fused): run-to-run identical
        if it % 5 == 0:
            rep, _ = V.run_device(eng, cfg, frames, vs, split=False)
            ref = got if not split else again
            nr = sum(V.canonical(*x) != V.canonical(*y) for x, y in zip(rep, ref))
            tot["not_repeatable"] += nr
            if nr:
                bad.append(dict(it=it, not_repeatable=nr))
    tot["worst_err_over_bound"] = round(tot["worst_err_over_bound"], 4)
    tot["seconds"] = round(time.time() - t0, 1)
    print(json.dumps({"seed": seed, "voxel": tot, "cloud_kinds": kinds, "first_bad": bad[:6]}))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
