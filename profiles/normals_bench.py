"""Point normals timing on device-resident clouds produced by the stage itself (480p density medium = the UI
default, 1080p medium and high; scene and uniform-random depth): median of CUDA-event times around
estimate_normals (bounds pass + grid build + query) after warm-up, k = 30 in k-NN mode and in radius mode, with the
shared-memory and the local-memory heap; beside it, on the same cloud, statistical outlier removal (same grid build,
k = 20) and the CPU oracle (scipy cKDTree on all host cores + Open3D's covariance and FastEigen3x3 in NumPy).
    python profiles/normals_bench.py [--no-cpu]        (one JSON line)"""
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import image_to_pointcloud_b200 as m  # noqa: E402
from profiles.voxel_sweep import depth_maps  # noqa: E402

RADIUS = 0.05   # stage units (depth_scale 10): ~30 neighbours at 1080p high near the middle of the scene


def timed(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(2):   # allocator and first-launch warm-up
        fn()
    torch.cuda.synchronize()
    per_call = []
    for _ in range(iters):
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        per_call.append(a.elapsed_time(b))
    return sorted(per_call)[len(per_call) // 2]


def card():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        out["power_limit_and_max_sm_clock"] = q
    except Exception as e:  # the numbers still stand with the card's name
        out["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return out


def bench(iters=9, cpu=True):
    dev = torch.device("cuda", 0)
    out = {}
    for name, (H, W, dens) in {"480p_medium": (480, 640, "medium"), "1080p_medium": (1080, 1920, "medium"),
                               "1080p_high": (1080, 1920, "high")}.items():
        maps, g = depth_maps(dev, H, W)
        bgr = torch.randint(0, 256, (1, H, W, 3), generator=g, device=dev, dtype=torch.uint8)
        eng = m.FrameEngine(H, W, batch=1, device=dev)
        cfg = eng.make_config(density=dens)
        for kind, depth in maps.items():
            res = eng.process(cfg, depth, bgr)
            n = int(res.count.cpu()[0])
            xyz, rgb = res.xyz[0, :n].contiguous(), res.rgb[0, :n].contiguous()
            row = {"points": n}
            for heap in ("shared", "local"):
                os.environ["D2PC_NORMALS_HEAP"] = heap   # read by every d2pc_normals_enqueue
                ms = timed(lambda: m.estimate_normals(xyz, knn=30, return_device=True), iters)
                row[f"knn30_{heap}_heap_ms"] = round(ms, 3)
            os.environ.pop("D2PC_NORMALS_HEAP")
            row["knn30_mpoints_per_s"] = round(n / min(row["knn30_shared_heap_ms"], row["knn30_local_heap_ms"]) / 1e3, 1)
            row[f"radius{RADIUS}_knn30_ms"] = round(timed(lambda: m.estimate_normals(xyz, knn=30, radius=RADIUS,
                                                                                   return_device=True), iters), 3)
            row["knn30_with_covariances_ms"] = round(timed(lambda: m.estimate_normals(
                xyz, knn=30, return_covariances=True, return_device=True), iters), 3)
            row["sor_k20_ms"] = round(timed(lambda: m.statistical_outlier_removal(xyz, rgb, return_device=True), iters), 3)
            if cpu and (name != "1080p_high" or kind == "scene"):
                from oracle import d2pc_normals_oracle as N
                pts = xyz.cpu().numpy()
                t0 = time.perf_counter()
                N.estimate_normals(pts, knn=30, workers=-1)
                row["cpu_oracle_all_cores_s"] = round(time.perf_counter() - t0, 3)
                row["cpu_cores"] = os.cpu_count()
                row["speedup_vs_cpu_oracle"] = round(row["cpu_oracle_all_cores_s"] * 1e3 / row["knn30_shared_heap_ms"], 1)
            out[f"{name}_{kind}"] = row
            print(f"{name}_{kind}", row, file=sys.stderr)
    return out


if __name__ == "__main__":
    print(json.dumps({"workload": "estimate_normals k=30 (k-NN and radius mode) on the stage's own clouds "
                                  "(scene / uniform-random depth), beside SOR k=20 and the CPU oracle",
                      "card": card(), "normals": bench(cpu="--no-cpu" not in sys.argv)}))
