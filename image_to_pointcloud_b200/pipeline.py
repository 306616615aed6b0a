"""Everything process_image_pipeline does between the depth network and the job result
(reference backend/app.py:468-559) in ONE device-resident pass:

    depth_to_point_cloud (:468-476) -> refine_point_cloud (:479)
    [-> remove_small_clusters of the refined rows (row f5), with cluster_eps] -> preview decimation (:495-506)
    -> save_point_cloud (:537) -> generate_gis_metadata bounds (:393-400)
    [-> estimate_normals, the mesh builder's first step (:271-308), with normals=True]
    [-> grid_mesh of the refined lattice rows, the mesh PLY (row m1), with mesh=True]
    [-> remove_small_components of that mesh (row m3), with mesh_min_triangles]
    [-> filter_smooth_taubin and compute_vertex_normals of that mesh (row m4), with mesh_smooth_iterations]
    [-> simplify_mesh of that mesh, the preview mesh PLY (row m2), with mesh_preview_voxel]

Called as separate drop-ins, those steps move the cloud across PCIe five times (down after the stage, up
and down around the refinement, up again for the writer).  Here the image and the depth map go up once,
every step runs on the rows where the previous one left them, and only what the caller keeps comes
down: the refined arrays (optional), the ~20 000 preview rows, the file bytes and six bounds.
Each step is the same kernel sequence the individual drop-ins use, so the results are identical.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path
from typing import Optional

import numpy as np
import torch

from . import _lib, cluster, writers
from ._lib import check
from .api import _engine_for, _image_channels, _to_host, bounds_dict, check_depth_dtype
from .engine import DENSITY_STEP
from .mesh import (_cos2, _max_edge, _small_components, check_iterations, check_min_triangles, check_voxel_size,
                   compute_vertex_normals, filter_smooth_taubin, grid_mesh, lattice_shape, simplify_mesh)
from .normals import estimate_normals
from .refine import statistical_outlier_removal


def point_cloud_stage(image: np.ndarray, depth: np.ndarray, *, density: str = "medium", invert: bool = True,
                      depth_scale: float = 10.0, smooth: bool = False, smooth_ksize: int = 5, fov: Optional[float] = None,
                      refine: bool = True, nb_neighbors: int = 20, std_ratio: float = 2.0,
                      output_format: Optional[str] = "ply", filename: Optional[str] = None,
                      max_preview: int = writers.MAX_PREVIEW, return_arrays: bool = True, normals: bool = False,
                      normals_knn: int = 30, mesh: bool = False, mesh_max_angle: float = 85.0, mesh_max_edge=None,
                      mesh_preview_voxel: Optional[float] = None, mesh_min_triangles: Optional[int] = None,
                      mesh_smooth_iterations: Optional[int] = None, cluster_eps: Optional[float] = None,
                      cluster_min_points: int = 10, cluster_min_size: int = 1, device=None) -> dict:
    """Returns a dict with ``points`` / ``colors`` (host float32 [M,3], if ``return_arrays``), ``point_count``,
    ``preview_points`` / ``preview_colors`` (nested lists as app.py:505-506), ``bounds`` (app.py:393-400),
    and either ``filepath`` (``filename`` given: the file the reference's writer would have put into
    outputs/<filename>.<ext>) or ``file_bytes`` (its content).  With ``normals`` the refined rows' normals
    (``estimate_normals(points, knn=normals_knn)``, float64 [M,3]) are computed on the device, returned as
    ``normals`` (if ``return_arrays``) and written into a PLY file.  With ``mesh`` the (refined) lattice rows are
    also meshed (``grid_mesh(..., max_angle=mesh_max_angle, max_edge=mesh_max_edge)``, vertex normals included):
    ``mesh_vertex_count``, ``mesh_triangle_count`` and either ``mesh_filepath`` (outputs/<filename>_mesh.ply) or
    ``mesh_file_bytes``.  With ``mesh_min_triangles`` (needs ``mesh``) the components of fewer triangles are removed
    from that mesh before it is written (``remove_small_components``): ``mesh_component_count`` (before the removal)
    and ``mesh_removed_triangle_count``, the counts above describing the cleaned mesh.  With
    ``mesh_smooth_iterations`` (needs ``mesh``) that mesh is then smoothed (``filter_smooth_taubin(mesh, N, 0.5, -0.53,
    scope="vertex")``) and its vertex normals recomputed (``compute_vertex_normals``) before it is written; 0 keeps
    the positions and still recomputes the normals.  With ``mesh_preview_voxel`` (needs ``mesh``) that (cleaned,
    smoothed) mesh is also simplified for a preview (``simplify_mesh(mesh, mesh_preview_voxel)``, average
    contraction): ``mesh_preview_vertex_count``,
    ``mesh_preview_triangle_count`` and either ``mesh_preview_filepath`` (outputs/<filename>_mesh_preview.ply) or
    ``mesh_preview_file_bytes``.  With ``cluster_eps`` the (refined) rows are clustered (``remove_small_clusters(
    points, colors, eps=cluster_eps, min_points=cluster_min_points, min_size=cluster_min_size)``) before the normals,
    the preview, the file, the bounds and the mesh: noise and clusters below ``cluster_min_size`` points are dropped
    from all of them (the mesh's lattice keep mask composes both removals).  It adds ``cluster_count`` (before the
    removal) and ``cluster_removed_point_count``."""
    DENSITY_STEP[density]  # KeyError first, like the reference
    if mesh:   # mesh argument errors before any device work
        _cos2(mesh_max_angle), _max_edge(mesh_max_edge)
    if mesh_preview_voxel is not None:
        if not mesh:
            raise ValueError("mesh_preview_voxel needs mesh=True")
        check_voxel_size(mesh_preview_voxel)
    if mesh_min_triangles is not None:
        if not mesh:
            raise ValueError("mesh_min_triangles needs mesh=True")
        check_min_triangles(mesh_min_triangles)
    if mesh_smooth_iterations is not None:
        if not mesh:
            raise ValueError("mesh_smooth_iterations needs mesh=True")
        check_iterations(mesh_smooth_iterations)
    if cluster_eps is not None:
        cluster_eps = cluster.check_eps(cluster_eps, "cluster_eps")
        cluster_min_points = cluster.check_min_points(cluster_min_points, "cluster_min_points")
        cluster_min_size = cluster.check_min_size(cluster_min_size, "cluster_min_size")
    lib = _lib.load_library()
    img_h, img_w = image.shape[:2]
    dep_h, dep_w = depth.shape[:2]
    check_depth_dtype(depth, int(img_h), int(img_w))
    img_c = _image_channels(image)
    eng = _engine_for(int(img_h), int(img_w), img_c, int(dep_h), int(dep_w), device)
    dev = eng.device
    cfg = eng.make_config(density=density, invert=invert, depth_scale=float(depth_scale), fov=fov)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev)
        d = torch.from_numpy(np.ascontiguousarray(depth, dtype=np.float32).reshape(1, dep_h, dep_w)).to(dev)
        im = torch.from_numpy(np.ascontiguousarray(image).reshape(1, img_h, img_w, -1)).to(dev) if img_c >= 3 else None
        res = eng.process(cfg, d, im, stream=stream, smooth_ksize=(smooth_ksize if smooth else None))
        n = int(res.count.cpu()[0])
        xyz, rgb = res.xyz[0, :n], res.rgb[0, :n]
        lat_xyz, lat_rgb, kept = xyz, rgb, None   # the emit rows are the unmasked lattice
        if refine and n > 0:
            xyz, rgb, kept, _ = statistical_outlier_removal(xyz, rgb, nb_neighbors, std_ratio, return_device=True)
        out = {}
        if cluster_eps is not None:
            r = cluster._run(xyz, rgb, cluster_eps, min_points=cluster_min_points, min_size=cluster_min_size)
            out["cluster_count"], out["cluster_removed_point_count"] = r["clusters"], int(xyz.shape[0]) - r["kept"]
            xyz, rgb = r["xyz"], r["rgb"]
            kept = r["index"] if kept is None else kept[r["index"].to(torch.int64)]
        m = int(xyz.shape[0])
        out["point_count"] = m
        nrm = estimate_normals(xyz, knn=normals_knn, return_device=True) if normals else None
        if return_arrays:
            out["points"], out["colors"] = _to_host(xyz), _to_host(rgb)   # pinned D2H at PCIe speed
            if normals:
                out["normals"] = nrm.cpu().numpy()
        pp, pc = writers.preview_lists(xyz, rgb, max_preview)
        out["preview_points"], out["preview_colors"] = pp, pc
        if m > 0:
            cnt = torch.tensor([m], dtype=torch.int32, device=dev)
            keys = torch.empty(6, dtype=torch.int32, device=dev)
            b6 = torch.empty(6, dtype=torch.float32, device=dev)
            check(lib.d2pc_rows_bounds_enqueue(xyz.data_ptr(), cnt.data_ptr(), m, keys.data_ptr(), b6.data_ptr(),
                                               stream.cuda_stream), "d2pc_rows_bounds_enqueue")
            out["bounds"] = bounds_dict(b6.cpu().numpy())
        fmt = (output_format or "").lower()
        if fmt:
            if fmt == "ply":
                rec = writers.ply_vertex_records(xyz, rgb, normals=nrm)
                header = writers.PLY_HEADER if nrm is None else writers.PLY_NORMAL_HEADER
                head, ext = header.format(n=len(rec)).encode("ascii"), "ply"
            elif fmt in ("las", "laz"):
                rec, offsets, mm = writers.las_point_records(xyz, rgb, 0.01)
                head, ext = writers.las_header(len(rec), 0.01, offsets, mm), "las"
            elif fmt == "xyz":
                rec, head, ext = np.frombuffer(writers.xyz_text(xyz, rgb), dtype=np.uint8), b"", "xyz"
            else:
                raise ValueError(f"Unsupported format: {output_format}")
            out["file_ext"] = ext
            if filename is not None:   # straight from the pinned buffer to the file, no concatenated copy
                Path("outputs").mkdir(exist_ok=True)
                path = f"outputs/{filename}.{ext}"
                with open(path, "wb") as f:
                    f.write(head)
                    f.write(memoryview(rec).cast("B"))
                out["filepath"] = path
            else:
                out["file_bytes"] = head + rec.tobytes()
        if mesh:
            keep = None
            if kept is not None:
                keep = torch.zeros(n, dtype=torch.uint8, device=dev)
                keep[kept.to(torch.int64)] = 1
            msh = grid_mesh(lat_xyz, lat_rgb, lattice_shape(img_h, img_w, density), keep=keep, max_edge=mesh_max_edge,
                            max_angle=mesh_max_angle, return_device=True)
            if mesh_min_triangles is not None:
                msh, out["mesh_component_count"], out["mesh_removed_triangle_count"] = _small_components(
                    msh, mesh_min_triangles, None, True, dev, True)
            if mesh_smooth_iterations is not None:
                msh = filter_smooth_taubin(msh, mesh_smooth_iterations, 0.5, -0.53, scope="vertex", return_device=True)
                msh = compute_vertex_normals(msh, return_device=True)
            out["mesh_vertex_count"], out["mesh_triangle_count"] = len(msh.vertices), len(msh.triangles)
            if filename is not None:
                out["mesh_filepath"] = writers.save_mesh_ply(msh, f"{filename}_mesh")
            else:
                out["mesh_file_bytes"] = writers.mesh_ply_bytes(msh)
            if mesh_preview_voxel is not None:
                pre = simplify_mesh(msh, mesh_preview_voxel, return_device=True)
                out["mesh_preview_vertex_count"] = len(pre.vertices)
                out["mesh_preview_triangle_count"] = len(pre.triangles)
                if filename is not None:
                    out["mesh_preview_filepath"] = writers.save_mesh_ply(pre, f"{filename}_mesh_preview")
                else:
                    out["mesh_preview_file_bytes"] = writers.mesh_ply_bytes(pre)
        return out
