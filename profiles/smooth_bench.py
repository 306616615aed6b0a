"""Mesh smoothing (row m4) timing on lattice meshes of the stage: 480p medium, 1080p medium, 1080p high and 4K high,
scene depth (depth_scale 10), each meshed by grid_mesh with normals.  Per case, medians of CUDA-event times after
warm-up, with L2 overwritten (256 MB memset) before every timed call:
  taubin1 / taubin10   d2pc_mesh_smooth_enqueue alone on preallocated buffers, Taubin with 1 and 10 iterations
                       (2 and 20 passes), scope "vertex" as the stage runs it
  per pass             (taubin10 - taubin1) / 18; adjacency build = taubin1 - 2 passes (both derived, not timed alone)
  call                 filter_smooth_taubin(mesh, 10, scope="vertex") on device tensors (allocations, one read-back)
  normals call         compute_vertex_normals(mesh) on device tensors
A pass needs at least 8 B of offsets, 4 B per adjacency entry, 24 B of float64 state read and 24 B written per vertex;
that over the per-pass time is compared with the 6451.8 GB/s copy peak DESIGN.md uses, and the two float64 states
(48 B per vertex) are compared with the 126 MB L2.  Beside it, the NumPy oracle (oracle/d2pc_smooth_oracle.py) on one
host core for Taubin x 10 (not run at 4K), with its equality to the device result.
    python profiles/smooth_bench.py [--no-cpu]        (one JSON line)"""
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
from oracle import d2pc_smooth_oracle as SMO  # noqa: E402  (entry count and the oracle beside the timing)
from profiles.voxel_sweep import depth_maps  # noqa: E402

L2_BYTES = 126e6


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
        _lib.check(lib.d2pc_mesh_smooth_scratch_bytes(V, T, C.byref(nb)), "scratch")
        scratch = torch.empty(nb.value, dtype=torch.uint8, device=dev)
        oxyz = torch.empty((V, 3), dtype=torch.float32, device=dev)
        orgb = torch.empty((V, 3), dtype=torch.float32, device=dev)
        onrm = torch.empty((V, 3), dtype=torch.float64, device=dev)
        err = torch.zeros(1, dtype=torch.int32, device=dev)

        def kernels(iterations):
            _lib.check(lib.d2pc_mesh_smooth_enqueue(
                mesh.vertices.data_ptr(), mesh.colors.data_ptr(), mesh.vertex_normals.data_ptr(), V,
                mesh.triangles.data_ptr(), T, _lib.SMOOTH_TAUBIN, iterations, 0.5, -0.53, _lib.SMOOTH_VERTEX,
                scratch.data_ptr(), scratch.numel(), oxyz.data_ptr(), orgb.data_ptr(), onrm.data_ptr(),
                err.data_ptr(), s), "d2pc_mesh_smooth_enqueue")
        t1 = timed(lambda: kernels(1), iters, flush)
        t10 = timed(lambda: kernels(10), iters, flush)
        e = int(err.cpu())
        call_ms = timed(lambda: m.filter_smooth_taubin(mesh, 10, scope="vertex", return_device=True), iters, flush)
        nrm_ms = timed(lambda: m.compute_vertex_normals(mesh, return_device=True), iters, flush)
        per_pass = (t10 - t1) / 18
        host = m.TriangleMesh(*(t.cpu().numpy() for t in mesh))
        E = int(SMO.adjacency(V, host.triangles)[0][-1])
        algo = 8 * V + 4 * E + 48 * V
        row = {"lattice": [R, Cc], "vertices": V, "triangles": T, "adjacency_entries": E, "error": e,
               "taubin1_kernels_ms": round(t1, 4), "taubin10_kernels_ms": round(t10, 4),
               "per_pass_ms": round(per_pass, 4), "adjacency_build_ms": round(t1 - 2 * per_pass, 4),
               "taubin10_call_ms": round(call_ms, 4), "compute_vertex_normals_call_ms": round(nrm_ms, 4),
               "pass_algorithmic_bytes": algo, "pass_achieved_gbs": round(algo / per_pass / 1e6, 1),
               "pass_fraction_of_copy_peak": round(algo / per_pass / 1e6 / PEAK_GBS, 4),
               "state_bytes": 48 * V, "state_fits_l2": 48 * V <= L2_BYTES}
        if cpu and name != "4k_high":
            kernels(10)
            got = oxyz.cpu().numpy()
            t0 = time.perf_counter()
            want = SMO.filter_smooth_taubin(host, 10, scope="vertex")
            row["oracle_taubin10_s"] = round(time.perf_counter() - t0, 3)
            row["oracle_equal"] = want.vertices.tobytes() == got.tobytes()
        out[name] = row
        print(name, row, file=sys.stderr)
        del scratch, oxyz, orgb, onrm, mesh, eng
        torch.cuda.empty_cache()
    return out


if __name__ == "__main__":
    print(json.dumps({"workload": "filter_smooth_taubin(10, scope=vertex) and compute_vertex_normals of grid_mesh "
                                  "lattice meshes (normals on) of the stage, scene depth, depth_scale 10; L2 "
                                  "overwritten before every timed call",
                      "card": card(), "peak_gbs": PEAK_GBS, "smooth": bench(cpu="--no-cpu" not in sys.argv)}))
