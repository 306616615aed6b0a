"""ctypes binding of libd2pc.so (include/d2pc.h).  No fallback: if the CUDA library is missing
or does not load, importing the product path fails loudly."""
from __future__ import annotations

import ctypes as C
import os

from .build import LIB_PATH, build_library

D2PC_ABI_VERSION = 1
D2PC_OK = 0
FRAME_PENDING, FRAME_READY, FRAME_NEEDS_FALLBACK = 0, 1, 2
BRANCH_PCT, BRANCH_MINMAX, BRANCH_ZEROS = 0, 1, 2
PATH_GRAPH, PATH_NO_OVERLAP, PATH_NO_L2_HINTS, PATH_ORDERED = 1, 2, 4, 8
MESH_REMOVE_UNREFERENCED, MESH_NORMALS = 1, 2
SIMPLIFY_QUADRIC, SIMPLIFY_NORMALS = 1, 2
SMOOTH_SIMPLE, SMOOTH_LAPLACIAN, SMOOTH_TAUBIN = 0, 1, 2
SMOOTH_VERTEX, SMOOTH_NORMAL, SMOOTH_COLOR = 1, 2, 4
CLUSTER_ERR_NONFINITE, CLUSTER_ERR_GRID, CLUSTER_ERR_BOUND = 1, 2, 4

EXPORTS = [
    "d2pc_abi_version", "d2pc_error_string", "d2pc_last_cuda_error", "d2pc_workspace_bytes",
    "d2pc_stats_enqueue", "d2pc_stats_fallback_enqueue", "d2pc_frame_status", "d2pc_frame_params",
    "d2pc_emit_enqueue", "d2pc_smooth_scratch_bytes", "d2pc_emit_smooth_enqueue",
    "d2pc_preview_enqueue", "d2pc_voxel_table_bytes", "d2pc_voxel_table_init", "d2pc_voxel_enqueue",
    "d2pc_preview_rows_enqueue", "d2pc_xyz_text_scratch_bytes", "d2pc_xyz_text_measure_enqueue",
    "d2pc_xyz_text_write_enqueue", "d2pc_rows_bounds_enqueue", "d2pc_las_records_enqueue", "d2pc_ply_records_enqueue", "d2pc_sor_scratch_bytes", "d2pc_sor_enqueue",
    "d2pc_ply_normal_records_enqueue", "d2pc_normals_scratch_bytes", "d2pc_normals_enqueue",
    "d2pc_grid_mesh_scratch_bytes", "d2pc_grid_mesh_enqueue", "d2pc_ply_face_records_enqueue",
    "d2pc_mesh_simplify_scratch_bytes", "d2pc_mesh_simplify_enqueue",
    "d2pc_mesh_components_scratch_bytes", "d2pc_mesh_components_enqueue", "d2pc_mesh_filter_scratch_bytes",
    "d2pc_mesh_filter_enqueue", "d2pc_mesh_smooth_scratch_bytes", "d2pc_mesh_smooth_enqueue",
    "d2pc_mesh_vertex_normals_scratch_bytes", "d2pc_mesh_vertex_normals_enqueue",
    "d2pc_cluster_scratch_bytes", "d2pc_radius_outlier_enqueue", "d2pc_dbscan_enqueue",
    "d2pc_path_create", "d2pc_path_destroy", "d2pc_path_enqueue", "d2pc_path_trace_offset",
]


class D2pcConfig(C.Structure):
    _fields_ = [
        ("batch", C.c_int32), ("img_h", C.c_int32), ("img_w", C.c_int32), ("img_c", C.c_int32),
        ("dep_h", C.c_int32), ("dep_w", C.c_int32), ("step", C.c_int32), ("invert", C.c_int32),
        ("depth_scale", C.c_double), ("cx", C.c_double), ("cy", C.c_double), ("f", C.c_double),
        ("use_z_range", C.c_int32), ("z_min", C.c_float), ("z_max", C.c_float),
        ("drop_nonfinite", C.c_int32), ("want_bounds", C.c_int32), ("force_fallback", C.c_int32),
    ]


class D2pcFrameParams(C.Structure):
    _fields_ = [
        ("p2", C.c_double), ("p98", C.c_double), ("den", C.c_double), ("inv_den", C.c_double),
        ("lo32", C.c_float), ("hi32", C.c_float), ("den32", C.c_float), ("median", C.c_float),
        ("branch", C.c_int32), ("status", C.c_int32), ("n_nonfinite", C.c_uint32), ("n_nan", C.c_uint32),
        ("n_cand", C.c_uint32 * 2), ("reserved", C.c_uint32 * 2),
    ]


class D2pcError(RuntimeError):
    def __init__(self, code: int, where: str, detail: str = ""):
        self.code = code
        super().__init__(f"{where} failed: {detail} (code {code})")


_lib = None


def load_library(path: str | None = None) -> C.CDLL:
    """Load (building first if the in-tree .so is stale or absent and nvcc is available)."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or os.environ.get("D2PC_LIBRARY") or None   # measurement aid: A/B runs against another build
    p = path or LIB_PATH
    if path is None:
        try:
            p = build_library()
        except Exception as e:
            # No compiler on this box (or the build failed).  A library built from exactly these sources is
            # fine; a stale one is not: tests and benchmarks would silently report against old kernels.
            from .build import source_digest, stored_digest
            if not os.path.exists(LIB_PATH):
                raise
            have, want = stored_digest(), source_digest()
            if have != want:
                raise RuntimeError(f"libd2pc.so is stale (built from sources {have}, tree is {want}) and could not "
                                   f"be rebuilt: {e}") from e
            p = LIB_PATH
    lib = C.CDLL(p)
    vp = C.c_void_p
    cfgp = C.POINTER(D2pcConfig)
    lib.d2pc_abi_version.restype = C.c_int
    lib.d2pc_error_string.restype = C.c_char_p
    lib.d2pc_error_string.argtypes = [C.c_int]
    lib.d2pc_last_cuda_error.restype = C.c_char_p
    lib.d2pc_workspace_bytes.argtypes = [cfgp, C.POINTER(C.c_size_t)]
    lib.d2pc_stats_enqueue.argtypes = [cfgp, vp, vp, C.c_size_t, vp]
    lib.d2pc_stats_fallback_enqueue.argtypes = [cfgp, vp, vp, C.c_size_t, vp]
    lib.d2pc_frame_status.argtypes = [cfgp, vp, vp, vp, vp]
    lib.d2pc_frame_params.argtypes = [cfgp, vp, vp, vp]
    lib.d2pc_emit_enqueue.argtypes = [cfgp, vp, vp, vp, C.c_size_t, vp, vp, vp, vp, vp]
    lib.d2pc_smooth_scratch_bytes.argtypes = [cfgp, C.POINTER(C.c_size_t)]
    lib.d2pc_emit_smooth_enqueue.argtypes = [cfgp, vp, vp, vp, C.c_size_t, C.c_int32, C.POINTER(C.c_double), vp,
                                             C.c_size_t, vp, vp, vp, vp, vp]
    lib.d2pc_preview_enqueue.argtypes = [cfgp, vp, vp, C.c_size_t, vp, vp, vp]
    lib.d2pc_voxel_table_bytes.argtypes = [cfgp, C.POINTER(C.c_size_t)]
    lib.d2pc_voxel_table_init.argtypes = [cfgp, vp, C.c_size_t, vp]
    lib.d2pc_voxel_enqueue.argtypes = [cfgp, C.c_double, vp, vp, vp, vp, vp, C.c_size_t, vp, vp, vp, vp, vp, vp]
    lib.d2pc_preview_rows_enqueue.argtypes = [vp, vp, vp, C.c_uint32, vp, vp, C.c_uint32, vp, vp]
    lib.d2pc_xyz_text_scratch_bytes.argtypes = [C.c_uint32, C.POINTER(C.c_size_t)]
    lib.d2pc_xyz_text_measure_enqueue.argtypes = [vp, vp, vp, C.c_uint32, vp, C.c_size_t, vp, vp, vp]
    lib.d2pc_xyz_text_write_enqueue.argtypes = [vp, vp, vp, C.c_uint32, vp, C.c_size_t, vp, vp, vp, C.c_size_t, vp]
    lib.d2pc_rows_bounds_enqueue.argtypes = [vp, vp, C.c_uint32, vp, vp, vp]
    lib.d2pc_las_records_enqueue.argtypes = [vp, vp, vp, C.c_uint32, vp, C.c_double, vp, vp, vp, vp]
    lib.d2pc_ply_records_enqueue.argtypes = [vp, vp, vp, C.c_uint32, vp, vp]
    lib.d2pc_sor_scratch_bytes.argtypes = [C.c_uint32, C.POINTER(C.c_size_t)]
    lib.d2pc_sor_enqueue.argtypes = [vp, vp, vp, C.c_uint32, vp, C.c_int32, C.c_double, vp, C.c_size_t, vp, vp, vp, vp, vp, vp]
    lib.d2pc_ply_normal_records_enqueue.argtypes = [vp, vp, vp, vp, C.c_uint32, vp, vp]
    lib.d2pc_normals_scratch_bytes.argtypes = [C.c_uint32, C.POINTER(C.c_size_t)]
    lib.d2pc_normals_enqueue.argtypes = [vp, vp, C.c_uint32, vp, C.c_int32, C.c_double, C.c_int32,
                                         C.POINTER(C.c_double), vp, C.c_size_t, vp, vp, vp]
    lib.d2pc_grid_mesh_scratch_bytes.argtypes = [C.c_uint32, C.c_uint32, C.POINTER(C.c_size_t)]
    lib.d2pc_grid_mesh_enqueue.argtypes = [vp, vp, vp, C.c_uint32, C.c_uint32, C.c_double, C.c_double, C.c_uint32,
                                           vp, C.c_size_t, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.d2pc_ply_face_records_enqueue.argtypes = [vp, vp, C.c_uint32, vp, vp]
    lib.d2pc_mesh_simplify_scratch_bytes.argtypes = [C.c_uint32, C.c_uint32, C.POINTER(C.c_size_t)]
    lib.d2pc_mesh_simplify_enqueue.argtypes = [vp, vp, vp, vp, C.c_uint32, vp, C.c_uint32, C.c_double, C.c_uint32, vp,
                                               C.c_size_t, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.d2pc_mesh_components_scratch_bytes.argtypes = [C.c_uint32, C.c_uint32, C.POINTER(C.c_size_t)]
    lib.d2pc_mesh_components_enqueue.argtypes = [vp, C.c_uint32, vp, C.c_uint32, vp, C.c_size_t, vp, vp, vp, vp, vp,
                                                 vp]
    lib.d2pc_mesh_filter_scratch_bytes.argtypes = [C.c_uint32, C.c_uint32, C.POINTER(C.c_size_t)]
    lib.d2pc_mesh_filter_enqueue.argtypes = [vp, vp, vp, vp, C.c_uint32, vp, C.c_uint32, vp, C.c_uint32, vp,
                                             C.c_size_t, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.d2pc_mesh_smooth_scratch_bytes.argtypes = [C.c_uint32, C.c_uint32, C.POINTER(C.c_size_t)]
    lib.d2pc_mesh_smooth_enqueue.argtypes = [vp, vp, vp, C.c_uint32, vp, C.c_uint32, C.c_int, C.c_uint32, C.c_double,
                                             C.c_double, C.c_uint32, vp, C.c_size_t, vp, vp, vp, vp, vp]
    lib.d2pc_mesh_vertex_normals_scratch_bytes.argtypes = [C.c_uint32, C.c_uint32, C.POINTER(C.c_size_t)]
    lib.d2pc_mesh_vertex_normals_enqueue.argtypes = [vp, C.c_uint32, vp, C.c_uint32, vp, C.c_size_t, vp, vp, vp]
    lib.d2pc_cluster_scratch_bytes.argtypes = [C.c_uint32, C.POINTER(C.c_size_t)]
    lib.d2pc_radius_outlier_enqueue.argtypes = [vp, vp, vp, C.c_uint32, vp, C.c_int32, C.c_double, vp, C.c_size_t, vp,
                                                vp, vp, vp, vp]
    lib.d2pc_dbscan_enqueue.argtypes = [vp, vp, vp, C.c_uint32, vp, C.c_double, C.c_int32, C.c_uint32, vp, C.c_size_t,
                                        vp, vp, vp, vp, vp, vp, vp]
    lib.d2pc_path_trace_offset.argtypes = [cfgp, C.POINTER(C.c_size_t)]
    lib.d2pc_path_create.argtypes = [C.POINTER(vp)]
    lib.d2pc_path_destroy.argtypes = [vp]
    lib.d2pc_path_destroy.restype = None
    lib.d2pc_path_enqueue.argtypes = [vp, cfgp, vp, vp, vp, C.c_size_t, vp, vp, vp, vp, vp, vp, C.c_int32, C.c_int32,
                                      C.c_int32, vp]
    for name in EXPORTS:
        fn = getattr(lib, name)
        if name not in ("d2pc_error_string", "d2pc_last_cuda_error", "d2pc_path_destroy"):
            fn.restype = C.c_int
    if lib.d2pc_abi_version() != D2PC_ABI_VERSION:
        raise RuntimeError("libd2pc.so ABI version mismatch")
    if path is None:
        _lib = lib
    return lib


def check(code: int, where: str) -> None:
    if code != D2PC_OK:
        lib = load_library()
        detail = lib.d2pc_error_string(code).decode()
        if code == 3:
            detail += ": " + lib.d2pc_last_cuda_error().decode()
        raise D2pcError(code, where, detail)
