"""Lattice mesh (row m1) timing on the stage's own lattices: 480p medium (the UI default), 1080p medium and high, 4K
high; scene and uniform-random depth.  Per case, medians of CUDA-event times after warm-up, with L2 overwritten
(256 MB memset) before every timed call:
  kernels      d2pc_grid_mesh_enqueue alone on preallocated buffers (classify, vertex flags, scan, vertices with
               normals, triangles), remove_unreferenced on, max_angle 85
  grid_mesh    the Python call on device tensors (allocations + the count read-back included)
  end_to_end   depth_to_mesh(image, depth) from host arrays to host arrays (emit + mesh + copies)
  faces        d2pc_ply_face_records_enqueue of the kept triangles
Achieved bandwidth counts the algorithmic bytes (24 B read per lattice row, 52 B written per vertex: xyz, rgb, float64
normal, int32 row; 12 B per triangle) against the 6451.8 GB/s copy peak DESIGN.md uses.  Beside it, the NumPy oracle
(oracle/d2pc_mesh_oracle.py) on the same lattice, one host core.
    python profiles/mesh_bench.py [--no-cpu]        (one JSON line)"""
import ctypes as C
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import image_to_pointcloud_b200 as m  # noqa: E402
from image_to_pointcloud_b200 import _lib  # noqa: E402
from profiles.normals_bench import card  # noqa: E402
from profiles.voxel_sweep import depth_maps  # noqa: E402

PEAK_GBS = 6451.8
CASES = {"480p_medium": (480, 640, "medium"), "1080p_medium": (1080, 1920, "medium"),
         "1080p_high": (1080, 1920, "high"), "4k_high": (2160, 3840, "high")}


def timed(fn, iters, flush):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    per_call = []
    for _ in range(iters):
        flush.zero_()
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        per_call.append(a.elapsed_time(b))
    return sorted(per_call)[len(per_call) // 2]


def bench(iters=15, cpu=True):
    dev = torch.device("cuda", 0)
    lib = m.load_library()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    s = torch.cuda.current_stream(dev).cuda_stream
    cos2 = np.cos(np.radians(85.0)) ** 2
    out = {}
    for name, (H, W, dens) in CASES.items():
        maps, g = depth_maps(dev, H, W)
        bgr = torch.randint(0, 256, (1, H, W, 3), generator=g, device=dev, dtype=torch.uint8)
        eng = m.FrameEngine(H, W, batch=1, device=dev)
        cfg = eng.make_config(density=dens)
        R, Cc = m.mesh.lattice_shape(H, W, dens)
        n = R * Cc
        for kind, depth in maps.items():
            res = eng.process(cfg, depth, bgr)
            xyz, rgb = res.xyz[0, :n].contiguous(), res.rgb[0, :n].contiguous()
            nb = C.c_size_t(0)
            _lib.check(lib.d2pc_grid_mesh_scratch_bytes(R, Cc, C.byref(nb)), "scratch")
            scratch = torch.empty(nb.value, dtype=torch.uint8, device=dev)
            vx, vc = torch.empty((n, 3), device=dev), torch.empty((n, 3), device=dev)
            vr = torch.empty(n, dtype=torch.int32, device=dev)
            vn = torch.empty((n, 3), dtype=torch.float64, device=dev)
            tri = torch.empty((2 * (R - 1) * (Cc - 1), 3), dtype=torch.int32, device=dev)
            cnt = torch.zeros(2, dtype=torch.int32, device=dev)

            def kernels():
                _lib.check(lib.d2pc_grid_mesh_enqueue(xyz.data_ptr(), rgb.data_ptr(), None, R, Cc, 0.0, cos2, 3,
                                                      scratch.data_ptr(), scratch.numel(), vx.data_ptr(), vc.data_ptr(),
                                                      vr.data_ptr(), vn.data_ptr(), cnt.data_ptr(), tri.data_ptr(),
                                                      cnt.data_ptr() + 4, s), "d2pc_grid_mesh_enqueue")
            k_ms = timed(kernels, iters, flush)
            nv, nt = (int(v) for v in cnt.cpu())
            frec = torch.empty(max(nt, 1) * 13 + 16, dtype=torch.uint8, device=dev)
            f_ms = timed(lambda: lib.d2pc_ply_face_records_enqueue(tri.data_ptr(), cnt.data_ptr() + 4, max(nt, 1),
                                                                   frec.data_ptr(), s), iters, flush)
            g_ms = timed(lambda: m.grid_mesh(xyz, rgb, (R, Cc), return_device=True), iters, flush)
            img, dep = bgr[0].cpu().numpy(), depth[0].cpu().numpy()
            e_ms = timed(lambda: m.depth_to_mesh(img, dep, dens), max(5, iters // 3), flush)
            algo = 24 * n + 52 * nv + 12 * nt
            row = {"lattice": [R, Cc], "rows": n, "vertices": nv, "triangles": nt,
                   "triangles_kept_of_possible": round(nt / max(1, 2 * (R - 1) * (Cc - 1)), 4),
                   "kernels_ms": round(k_ms, 4), "kernels_grows_per_s": round(n / k_ms / 1e6, 2),
                   "algorithmic_bytes": algo, "achieved_gbs": round(algo / k_ms / 1e6, 1),
                   "fraction_of_copy_peak": round(algo / k_ms / 1e6 / PEAK_GBS, 3),
                   "face_records_ms": round(f_ms, 4), "grid_mesh_call_ms": round(g_ms, 4),
                   "depth_to_mesh_end_to_end_ms": round(e_ms, 3)}
            if cpu:
                from oracle import d2pc_mesh_oracle as MO
                hx, hr = xyz.cpu().numpy(), rgb.cpu().numpy()
                t0 = time.perf_counter()
                want = MO.grid_mesh(hx, hr, (R, Cc))
                row["numpy_oracle_s"] = round(time.perf_counter() - t0, 3)
                row["speedup_vs_numpy_oracle"] = round(row["numpy_oracle_s"] * 1e3 / k_ms, 1)
                got = m.grid_mesh(xyz, rgb, (R, Cc))
                row["bit_exact_vs_oracle"] = all(a.tobytes() == b.tobytes() for a, b in zip(got, want))
            out[f"{name}_{kind}"] = row
            print(f"{name}_{kind}", row, file=sys.stderr)
            del scratch, vx, vc, vr, vn, tri
        del eng
        torch.cuda.empty_cache()
    return out


if __name__ == "__main__":
    print(json.dumps({"workload": "grid_mesh (lattice mesh, normals on, max_angle 85, unreferenced removed) on the "
                                  "stage's own lattices, scene / uniform-random depth; L2 overwritten before every "
                                  "timed call", "card": card(), "peak_gbs": PEAK_GBS,
                      "mesh": bench(cpu="--no-cpu" not in sys.argv)}))
