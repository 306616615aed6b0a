"""Density clustering on the B200: cluster_dbscan / remove_small_clusters / remove_radius_outlier on the stage's own
clouds after statistical outlier removal (480p medium, 1080p medium, 1080p high, 4K high; scene and uniform-random
depth), eps 2x and 5x the median spacing, min_points 10.  Records the kernels alone (d2pc_dbscan_enqueue,
d2pc_radius_outlier_enqueue on device-resident rows) and the Python call, as medians of CUDA events with L2
overwritten (a 256 MB write) before each call, and the scipy oracle beside them where it finishes in reasonable time.
    python profiles/cluster_bench.py [out.json] [reps]        (one JSON line per configuration; the whole result
                                                               is written to out.json when it is given)"""
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import image_to_pointcloud_b200 as m  # noqa: E402
from image_to_pointcloud_b200 import _lib  # noqa: E402
from oracle import d2pc_cluster_oracle as CL  # noqa: E402  (checker and CPU timing only)
from tests import cases  # noqa: E402

FRAMES = [("480p", 480, 640, "medium"), ("1080p", 1080, 1920, "medium"), ("1080p", 1080, 1920, "high"),
          ("4K", 2160, 3840, "high")]
ORACLE_MAX_ROWS = 600_000


def median_spacing(p):
    from scipy.spatial import cKDTree
    q = p.astype(np.float64)
    d, _ = cKDTree(q).query(q, k=2, workers=-1)
    return float(np.median(d[:, 1]))


def timed(fn, reps, flush):
    ts = []
    for _ in range(reps):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def kernels(lib, xyz, rgb, eps, min_points, radius_mode):
    n = xyz.shape[0]
    nb = C.c_size_t(0)
    lib.d2pc_cluster_scratch_bytes(n, C.byref(nb))
    scratch = torch.empty(int(nb.value), dtype=torch.uint8, device="cuda")
    count = torch.tensor([n], dtype=torch.int32, device="cuda")
    keys = torch.empty(6, dtype=torch.int32, device="cuda")
    bounds = torch.empty(6, dtype=torch.float32, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    lib.d2pc_rows_bounds_enqueue(xyz.data_ptr(), count.data_ptr(), n, keys.data_ptr(), bounds.data_ptr(), s)
    labels = torch.empty(n, dtype=torch.int32, device="cuda")
    sizes = torch.empty(n, dtype=torch.int32, device="cuda")
    oxyz, orgb = torch.empty_like(xyz), torch.empty_like(rgb)
    oidx = torch.empty(n, dtype=torch.int32, device="cuda")
    counts = torch.zeros(4, dtype=torch.int32, device="cuda")

    def run():
        if radius_mode:
            rc = lib.d2pc_radius_outlier_enqueue(xyz.data_ptr(), rgb.data_ptr(), count.data_ptr(), n, bounds.data_ptr(),
                                                 min_points, eps, scratch.data_ptr(), scratch.numel(), oxyz.data_ptr(),
                                                 orgb.data_ptr(), oidx.data_ptr(), counts.data_ptr(), s)
        else:
            rc = lib.d2pc_dbscan_enqueue(xyz.data_ptr(), rgb.data_ptr(), count.data_ptr(), n, bounds.data_ptr(), eps,
                                         min_points, 1, scratch.data_ptr(), scratch.numel(), labels.data_ptr(),
                                         sizes.data_ptr(), oxyz.data_ptr(), orgb.data_ptr(), oidx.data_ptr(),
                                         counts.data_ptr(), s)
        assert rc == 0
    return run, counts


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 15
    lib = _lib.load_library()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    rows = []
    for name, H, W, density in FRAMES:
        for kind in ("scene", "uniform"):
            img, dep = cases.make_image(H, W, 1), cases.make_depth(H, W, 1, kind)
            p, c = m.depth_to_point_cloud(img, dep, density=density)
            p, c, _, _ = m.statistical_outlier_removal(p, c)
            h = median_spacing(p)
            xyz, rgb = torch.from_numpy(p).cuda(), torch.from_numpy(c).cuda()
            for f in (2.0, 5.0):
                eps = f * h
                rec = {"frame": name, "density": density, "depth": kind, "rows": len(p), "eps_factor": f,
                       "eps": eps, "min_points": 10}
                for mode in ("dbscan", "radius"):
                    run, counts = kernels(lib, xyz, rgb, eps, 10, mode == "radius")
                    run()
                    torch.cuda.synchronize()
                    rec[f"{mode}_kernels_ms"] = timed(run, reps, flush)
                    cnt = counts.cpu().numpy()
                    rec[f"{mode}_kept"] = int(cnt[0])
                    if mode == "dbscan":
                        rec["clusters"] = int(cnt[2])
                    assert cnt[1] == 0
                m.cluster_dbscan(xyz, eps, 10)
                rec["cluster_dbscan_call_ms"] = timed(lambda: m.cluster_dbscan(xyz, eps, 10, return_device=True),
                                                      reps, flush)
                rec["remove_small_clusters_call_ms"] = timed(
                    lambda: m.remove_small_clusters(xyz, rgb, eps=eps, min_points=10, return_device=True), reps, flush)
                rec["remove_radius_outlier_call_ms"] = timed(
                    lambda: m.remove_radius_outlier(xyz, rgb, nb_points=10, radius=eps, return_device=True), reps,
                    flush)
                if len(p) <= ORACLE_MAX_ROWS and f == 2.0:
                    t = time.perf_counter()
                    want = CL.cluster_dbscan(p, eps, 10)
                    rec["scipy_oracle_dbscan_s"] = time.perf_counter() - t
                    rec["equal_to_oracle"] = bool(np.array_equal(m.cluster_dbscan(p, eps, 10), want))
                rows.append(rec)
                print(json.dumps(rec), flush=True)
    res = {"gpu": gpu, "l2": "overwritten (256 MB write) before every timed call", "timing": "median of CUDA events",
           "reps": reps, "rows": rows}
    if out_path:
        os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
        with open(out_path, "w") as f:
            json.dump(res, f)
    print(json.dumps({"gpu": gpu, "configs": len(rows)}))


if __name__ == "__main__":
    main()
