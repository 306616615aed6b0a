"""Mesh components (row m3) timing on lattice meshes of the stage: 480p medium, 1080p medium, 1080p high and 4K high,
scene depth (depth_scale 10), each meshed by grid_mesh with normals.  Per case, medians of CUDA-event times after
warm-up, with L2 overwritten (256 MB memset) before every timed call:
  kernels        d2pc_mesh_components_enqueue alone on preallocated buffers
  call           cluster_connected_triangles on device tensors (allocations and the one read-back included)
  clean call     remove_small_components(min_triangles=10) on device tensors (both kernel calls, two read-backs)
Achieved bandwidth counts the algorithmic bytes of the components call (12 B of ids and 36 B of corner coordinates
read and 4 B of label written per triangle, 16 B written per cluster) against the 6451.8 GB/s copy peak DESIGN.md
uses.  Beside it, the NumPy / scipy oracle (oracle/d2pc_components_oracle.py) on one host core (not run at 4K).
    python profiles/components_bench.py [--no-cpu]        (one JSON line)"""
import ctypes as C
import json
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import image_to_pointcloud_b200 as m  # noqa: E402
from image_to_pointcloud_b200 import _lib  # noqa: E402
from profiles.mesh_bench import CASES, PEAK_GBS, timed  # noqa: E402
from profiles.normals_bench import card  # noqa: E402
from profiles.voxel_sweep import depth_maps  # noqa: E402


def bench(iters=11, cpu=True):
    dev = torch.device("cuda", 0)
    lib = m.load_library()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    s = torch.cuda.current_stream(dev).cuda_stream
    out = {}
    for name, (H, W, dens) in CASES.items():
        maps, g = depth_maps(dev, H, W)
        bgr = torch.randint(0, 256, (1, H, W, 3), generator=g, device=dev, dtype=torch.uint8)
        eng = m.FrameEngine(H, W, batch=1, device=dev)
        cfg = eng.make_config(density=dens)
        R, Cc = m.mesh.lattice_shape(H, W, dens)
        n = R * Cc
        res = eng.process(cfg, maps["scene"], bgr)
        mesh = m.grid_mesh(res.xyz[0, :n].contiguous(), res.rgb[0, :n].contiguous(), (R, Cc), return_device=True)
        V, T = len(mesh.vertices), len(mesh.triangles)
        nb = C.c_size_t(0)
        _lib.check(lib.d2pc_mesh_components_scratch_bytes(V, T, C.byref(nb)), "scratch")
        scratch = torch.empty(nb.value, dtype=torch.uint8, device=dev)
        lab = torch.empty(T, dtype=torch.int32, device=dev)
        cn = torch.empty(T, dtype=torch.int64, device=dev)
        ca = torch.empty(T, dtype=torch.float64, device=dev)
        words = torch.zeros(2, dtype=torch.int32, device=dev)

        def kernels():
            _lib.check(lib.d2pc_mesh_components_enqueue(
                mesh.vertices.data_ptr(), V, mesh.triangles.data_ptr(), T, scratch.data_ptr(), scratch.numel(),
                lab.data_ptr(), cn.data_ptr(), ca.data_ptr(), words.data_ptr(), words.data_ptr() + 4, s),
                "d2pc_mesh_components_enqueue")
        k_ms = timed(kernels, iters, flush)
        K, err = (int(v) for v in words.cpu())
        c_ms = timed(lambda: m.cluster_connected_triangles(mesh, return_device=True), iters, flush)
        r_ms = timed(lambda: m.remove_small_components(mesh, min_triangles=10, return_device=True), iters, flush)
        algo = 52 * T + 16 * K
        sizes = cn[:K]
        row = {"lattice": [R, Cc], "vertices": V, "triangles": T, "clusters": K, "error": err,
               "largest_cluster": int(sizes.max()) if K else 0,
               "clusters_below_10": int((sizes < 10).sum()), "kernels_ms": round(k_ms, 4),
               "triangles_per_s_g": round(T / k_ms / 1e6, 3), "algorithmic_bytes": algo,
               "achieved_gbs": round(algo / k_ms / 1e6, 1),
               "fraction_of_copy_peak": round(algo / k_ms / 1e6 / PEAK_GBS, 4),
               "cluster_connected_triangles_call_ms": round(c_ms, 4),
               "remove_small_components_call_ms": round(r_ms, 4)}
        if cpu and name != "4k_high":
            from oracle import d2pc_components_oracle as CO
            host = m.TriangleMesh(*(t.cpu().numpy() for t in mesh))
            t0 = time.perf_counter()
            want = CO.cluster_connected_triangles(host)
            row["oracle_s"] = round(time.perf_counter() - t0, 3)
            row["oracle_equal"] = all(a.tobytes() == b.cpu().numpy().tobytes()
                                      for a, b in zip(want, (lab, cn[:K], ca[:K])))
        out[name] = row
        print(name, row, file=sys.stderr)
        del scratch, lab, cn, ca, mesh, eng
        torch.cuda.empty_cache()
    return out


if __name__ == "__main__":
    print(json.dumps({"workload": "cluster_connected_triangles of grid_mesh lattice meshes (normals on) of the stage, "
                                  "scene depth, depth_scale 10; L2 overwritten before every timed call",
                      "card": card(), "peak_gbs": PEAK_GBS, "components": bench(cpu="--no-cpu" not in sys.argv)}))
