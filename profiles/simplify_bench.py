"""Mesh simplification (row m2) timing on lattice meshes of the stage: 480p medium, 1080p medium, 1080p high and 4K
high, scene and uniform-random depth (depth_scale 10), each meshed by grid_mesh with normals, then simplified at voxel
sizes from just above the lattice spacing to 0.1, both contractions.  Per case, medians of CUDA-event times after
warm-up, with L2 overwritten (256 MB memset) before every timed call:
  kernels        d2pc_mesh_simplify_enqueue alone on preallocated buffers
  call           simplify_mesh on device tensors (allocations and the one read-back of counts and error included)
Achieved bandwidth counts the algorithmic bytes (56 B read per vertex: xyz, rgb, float64 normal, int64 row; 12 B per
triangle; the same per output vertex and triangle written) against the 6451.8 GB/s copy peak DESIGN.md uses.  Beside
it, the NumPy oracle (oracle/d2pc_simplify_oracle.py) on one host core for the 0.02 voxel of each lattice (not run at
4K, where it takes minutes).
    python profiles/simplify_bench.py [--no-cpu]        (one JSON line)"""
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
from profiles.mesh_bench import CASES, PEAK_GBS, timed  # noqa: E402
from profiles.normals_bench import card  # noqa: E402
from profiles.voxel_sweep import depth_maps  # noqa: E402

VOXELS = (0.003, 0.01, 0.02, 0.1)


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
        for kind, depth in maps.items():
            res = eng.process(cfg, depth, bgr)
            mesh = m.grid_mesh(res.xyz[0, :n].contiguous(), res.rgb[0, :n].contiguous(), (R, Cc), return_device=True)
            V, T = len(mesh.vertices), len(mesh.triangles)
            nb = C.c_size_t(0)
            _lib.check(lib.d2pc_mesh_simplify_scratch_bytes(V, T, C.byref(nb)), "scratch")
            scratch = torch.empty(nb.value, dtype=torch.uint8, device=dev)
            ox, oc = torch.empty((V, 3), device=dev), torch.empty((V, 3), device=dev)
            on = torch.empty((V, 3), dtype=torch.float64, device=dev)
            orow = torch.empty(V, dtype=torch.int64, device=dev)
            otri = torch.empty((max(T, 1), 3), dtype=torch.int32, device=dev)
            words = torch.zeros(3, dtype=torch.int32, device=dev)
            rows = mesh.vertex_rows.contiguous()
            host = None
            for vs in VOXELS:
                for contraction in ("average", "quadric"):
                    flags = 2 | (1 if contraction == "quadric" else 0)

                    def kernels():
                        _lib.check(lib.d2pc_mesh_simplify_enqueue(
                            mesh.vertices.data_ptr(), mesh.colors.data_ptr(), mesh.vertex_normals.data_ptr(),
                            rows.data_ptr(), V, mesh.triangles.data_ptr(), T, vs, flags, scratch.data_ptr(),
                            scratch.numel(), ox.data_ptr(), oc.data_ptr(), on.data_ptr(), orow.data_ptr(),
                            words.data_ptr(), otri.data_ptr(), words.data_ptr() + 4, words.data_ptr() + 8, s),
                            "d2pc_mesh_simplify_enqueue")
                    k_ms = timed(kernels, iters, flush)
                    kv, kt, err = (int(v) for v in words.cpu())
                    c_ms = timed(lambda: m.simplify_mesh(mesh, vs, contraction=contraction, return_device=True),
                                 iters, flush)
                    algo = 56 * V + 12 * T + 56 * kv + 12 * kt
                    row = {"lattice": [R, Cc], "vertices_in": V, "triangles_in": T, "vertices_out": kv,
                           "triangles_out": kt, "error": err, "kernels_ms": round(k_ms, 4),
                           "vertices_per_s_g": round(V / k_ms / 1e6, 3), "algorithmic_bytes": algo,
                           "achieved_gbs": round(algo / k_ms / 1e6, 1),
                           "fraction_of_copy_peak": round(algo / k_ms / 1e6 / PEAK_GBS, 4),
                           "simplify_mesh_call_ms": round(c_ms, 4)}
                    if cpu and vs == 0.02 and name != "4k_high":
                        from oracle import d2pc_simplify_oracle as SO
                        if host is None:
                            host = m.TriangleMesh(*(t.cpu().numpy() for t in mesh))
                        t0 = time.perf_counter()
                        want = SO.simplify_mesh(host, vs, contraction)
                        row["numpy_oracle_s"] = round(time.perf_counter() - t0, 3)
                        row["oracle_counts_equal"] = (len(want.vertices), len(want.triangles)) == (kv, kt)
                    out[f"{name}_{kind}_{vs}_{contraction}"] = row
                    print(f"{name}_{kind}_{vs}_{contraction}", row, file=sys.stderr)
            del scratch, ox, oc, on, orow, otri, mesh
        del eng
        torch.cuda.empty_cache()
    return out


if __name__ == "__main__":
    print(json.dumps({"workload": "simplify_mesh of grid_mesh lattice meshes (normals on) of the stage, scene / "
                                  "uniform-random depth, depth_scale 10; L2 overwritten before every timed call",
                      "card": card(), "peak_gbs": PEAK_GBS, "simplify": bench(cpu="--no-cpu" not in sys.argv)}))
