"""image_to_pointcloud_b200 -- B200 (sm_100a) implementation of one stage of
Samsonboadi/Image_to_pointCloud: predicted depth map -> coloured 3-D point cloud
(reference backend/app.py:174-250), behind the reference's own function signature.

    from image_to_pointcloud_b200 import depth_to_point_cloud      # drop-in for app.py:174

The package holds only what that path needs: ``csrc/`` (CUDA kernels + the C ABI declared in
``include/d2pc.h``), the ctypes binding, and the host-side mirror of the reference interface.
"""
from .api import create_depth_preview, depth_preview_bgr, depth_to_point_cloud, depth_to_point_cloud_batch
from .engine import DENSITY_STEP, BatchStream, EmitResult, FrameEngine, reference_intrinsics, shard_frames
from .hostpipe import HostFramePipeline, MultiGpuPipeline
from .cluster import cluster_dbscan, remove_radius_outlier, remove_small_clusters
from ._lib import D2pcConfig, D2pcError, D2pcFrameParams, load_library
from .mesh import (TriangleMesh, cluster_connected_triangles, compute_vertex_normals, depth_to_mesh,
                   filter_smooth_laplacian, filter_smooth_simple, filter_smooth_taubin, grid_mesh,
                   remove_small_components, remove_triangles_by_mask, simplify_mesh)
from .normals import estimate_normals
from .pipeline import point_cloud_stage
from .refine import refine_point_cloud, statistical_outlier_removal
from .writers import (las_point_records, mesh_ply_bytes, ply_face_records, ply_vertex_records, preview_lists,
                      preview_rows, save_las, save_mesh_ply, save_ply, save_point_cloud, save_xyz, xyz_text)

__all__ = [
    "depth_to_point_cloud", "depth_to_point_cloud_batch", "create_depth_preview", "depth_preview_bgr", "FrameEngine", "HostFramePipeline", "MultiGpuPipeline",
    "EmitResult", "BatchStream", "DENSITY_STEP", "reference_intrinsics", "shard_frames",
    "D2pcConfig", "D2pcFrameParams", "D2pcError", "load_library",
    "preview_rows", "preview_lists", "xyz_text", "save_xyz", "las_point_records", "save_las", "ply_vertex_records",
    "save_ply", "save_point_cloud", "refine_point_cloud", "statistical_outlier_removal", "point_cloud_stage",
    "estimate_normals", "grid_mesh", "depth_to_mesh", "TriangleMesh", "ply_face_records", "mesh_ply_bytes",
    "save_mesh_ply", "simplify_mesh", "cluster_connected_triangles", "remove_triangles_by_mask",
    "remove_small_components", "filter_smooth_simple", "filter_smooth_laplacian", "filter_smooth_taubin",
    "compute_vertex_normals", "cluster_dbscan", "remove_radius_outlier", "remove_small_clusters",
]
__version__ = "0.1.0"
