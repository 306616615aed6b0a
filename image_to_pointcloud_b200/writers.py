"""Row f3: the reference's preview decimation and point-cloud writers (backend/app.py:310-389, 495-506)
with the per-point work moved to the GPU.

    preview_lists(points, colors)            app.py:495-506   strided rows -> nested lists for the JSON
    save_xyz(points, colors, filename)       app.py:379-389   ASCII "%.6f %.6f %.6f %d %d %d" lines
    save_las(points, colors, filename)       app.py:343-377   LAS 1.2, point format 2 (scale 0.01, offset = min)
    save_ply(points, colors, filename)       app.py:329-341   Open3D binary little-endian PLY (normals=: with nx, ny, nz)
    save_mesh_ply(mesh, filename)            (row m1)         Open3D write_triangle_mesh binary PLY of a TriangleMesh
    save_point_cloud(points, colors, format, filename)   app.py:310-327   the dispatcher

Same signatures and return values (the file path under ``outputs/``) as the reference.  ``points`` /
``colors`` may be the NumPy arrays ``depth_to_point_cloud`` returned (they are uploaded once) or CUDA
tensors (rows of a ``FrameEngine`` result, nothing is re-uploaded).  The kernels of libd2pc.so produce
the exact bytes of every row; the host only writes headers and files.  No CPU formatting path exists.

Parity: the XYZ text is byte-identical to the reference's own ``save_xyz`` (golden file in
tests/golden/writers.npz).  LAS and PLY bodies follow laspy's / Open3D's published record layouts;
neither library is installed in the build container, so those two are "parity unpinned" (DESIGN.md).
"""
from __future__ import annotations

import ctypes as C
import datetime
import logging
import struct
from pathlib import Path
from typing import Optional, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import check

logger = logging.getLogger(__name__)

LAS_RECORD_BYTES = 26
PLY_RECORD_BYTES = 27
PLY_NORMAL_RECORD_BYTES = 51
PLY_FACE_RECORD_BYTES = 13
MAX_PREVIEW = 20000  # app.py:496


def _device_rows(points, colors, device=None):
    """-> (xyz [n,3] f32 cuda, rgb [n,3] f32 cuda, count int32 [1] cuda, n)"""
    if not torch.cuda.is_available():
        raise RuntimeError("image_to_pointcloud_b200 needs a CUDA device (no CPU fallback exists)")
    if isinstance(points, torch.Tensor):
        xyz = points
        dev = xyz.device
    else:
        dev = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        xyz = torch.from_numpy(np.ascontiguousarray(points, dtype=np.float32)).to(dev)
    n = int(xyz.shape[0])
    if colors is None or len(colors) != n:
        # the reference's writers fall back to grey when there are no colours (app.py:371-374, 386)
        rgb = torch.full((n, 3), 128.0, dtype=torch.float32, device=dev)
    elif isinstance(colors, torch.Tensor):
        rgb = colors.to(dev)
    else:
        rgb = torch.from_numpy(np.ascontiguousarray(colors, dtype=np.float32)).to(dev)
    if xyz.dtype != torch.float32 or rgb.dtype != torch.float32 or xyz.dim() != 2 or xyz.shape[1] != 3:
        raise ValueError("points / colors must be float32 [N, 3]")
    xyz, rgb = xyz.contiguous(), rgb.contiguous()
    count = torch.tensor([n], dtype=torch.int32, device=dev)
    return xyz, rgb, count, n


def _stream(dev) -> int:
    return torch.cuda.current_stream(dev).cuda_stream


# ---- preview (app.py:495-506) ----------------------------------------------------------------
def preview_rows(points, colors, max_preview: int = MAX_PREVIEW, device=None) -> Tuple[np.ndarray, np.ndarray]:
    """points[::stride], colors[::stride] with the reference's stride rule, gathered on the device so
    only the preview rows cross PCIe."""
    lib = _lib.load_library()
    xyz, rgb, count, n = _device_rows(points, colors, device)
    cap = max(1, min(n, 2 * max_preview + 1))
    with torch.cuda.device(xyz.device):
        oxyz = torch.empty((cap, 3), dtype=torch.float32, device=xyz.device)
        orgb = torch.empty((cap, 3), dtype=torch.float32, device=xyz.device)
        ocnt = torch.zeros(1, dtype=torch.int32, device=xyz.device)
        if n > 0:
            check(lib.d2pc_preview_rows_enqueue(xyz.data_ptr(), rgb.data_ptr(), count.data_ptr(), int(max_preview),
                                                oxyz.data_ptr(), orgb.data_ptr(), cap, ocnt.data_ptr(),
                                                _stream(xyz.device)), "d2pc_preview_rows_enqueue")
        m = int(ocnt.cpu()[0])
        return oxyz[:m].cpu().numpy(), orgb[:m].cpu().numpy()


def preview_lists(points, colors, max_preview: int = MAX_PREVIEW, device=None):
    """(preview_points, preview_colors) exactly as app.py:505-506 builds them."""
    p, c = preview_rows(points, colors, max_preview, device)
    return p.astype(float).tolist(), c.astype(float).tolist()


# ---- XYZ ASCII (app.py:379-389) ---------------------------------------------------------------
def xyz_text(points, colors, device=None) -> bytes:
    lib = _lib.load_library()
    xyz, rgb, count, n = _device_rows(points, colors, device)
    if n == 0:
        return b""
    dev = xyz.device
    with torch.cuda.device(dev):
        nbytes = C.c_size_t(0)
        check(lib.d2pc_xyz_text_scratch_bytes(n, C.byref(nbytes)), "d2pc_xyz_text_scratch_bytes")
        scratch = torch.empty(int(nbytes.value), dtype=torch.uint8, device=dev)
        total = torch.zeros(1, dtype=torch.int64, device=dev)
        err = torch.zeros(1, dtype=torch.int32, device=dev)
        check(lib.d2pc_xyz_text_measure_enqueue(xyz.data_ptr(), rgb.data_ptr(), count.data_ptr(), n,
                                                scratch.data_ptr(), scratch.numel(), total.data_ptr(),
                                                err.data_ptr(), _stream(dev)), "d2pc_xyz_text_measure_enqueue")
        if int(err.cpu()[0]) != 0:
            # the reference raises here as well (int(nan) / int(inf)); huge magnitudes are not supported
            raise ValueError("cannot format the point cloud as XYZ text (non-finite colour or |coordinate| >= 2^44)")
        size = int(total.cpu()[0])
        text = torch.empty(size + 16, dtype=torch.uint8, device=dev)
        check(lib.d2pc_xyz_text_write_enqueue(xyz.data_ptr(), rgb.data_ptr(), count.data_ptr(), n,
                                              scratch.data_ptr(), scratch.numel(), total.data_ptr(), err.data_ptr(),
                                              text.data_ptr(), size, _stream(dev)), "d2pc_xyz_text_write_enqueue")
        host = torch.empty(size, dtype=torch.uint8, pin_memory=True)
        host.copy_(text[:size])
        return host.numpy().tobytes()


def save_xyz(points, colors, filename: str, device=None) -> str:
    """Save as XYZ ASCII format (reference save_xyz, app.py:379-389)."""
    filepath = f"outputs/{filename}.xyz"
    data = xyz_text(points, colors, device)
    with open(filepath, "wb") as f:
        f.write(data)
    return filepath


# ---- LAS 1.2 point format 2 (app.py:343-377) --------------------------------------------------
def las_point_records(points, colors, scale: float = 0.01, offsets=None, device=None):
    """-> (records uint8 [n, 26], offsets [3] float, int_minmax int32 [6])."""
    lib = _lib.load_library()
    xyz, rgb, count, n = _device_rows(points, colors, device)
    if n == 0:
        raise ValueError("No points to write to LAS")
    dev = xyz.device
    with torch.cuda.device(dev):
        bounds = torch.zeros(6, dtype=torch.float32, device=dev)
        if offsets is None:  # float(points[:, k].min()), app.py:352
            keys = torch.empty(6, dtype=torch.int32, device=dev)
            check(lib.d2pc_rows_bounds_enqueue(xyz.data_ptr(), count.data_ptr(), n, keys.data_ptr(), bounds.data_ptr(),
                                               _stream(dev)), "d2pc_rows_bounds_enqueue")
            offsets = [float(v) for v in bounds[:3].cpu()]
        else:
            bounds[:3] = torch.tensor([float(v) for v in offsets], dtype=torch.float32)
        rec = torch.empty(n * LAS_RECORD_BYTES + 16, dtype=torch.uint8, device=dev)
        mm = torch.zeros(6, dtype=torch.int32, device=dev)
        err = torch.zeros(1, dtype=torch.int32, device=dev)
        check(lib.d2pc_las_records_enqueue(xyz.data_ptr(), rgb.data_ptr(), count.data_ptr(), n, bounds.data_ptr(),
                                           float(scale), rec.data_ptr(), mm.data_ptr(), err.data_ptr(), _stream(dev)),
              "d2pc_las_records_enqueue")
        if int(err.cpu()[0]) != 0:
            raise OverflowError("LAS: scaled coordinate does not fit int32 (laspy raises OverflowError here)")
        host = torch.empty(n * LAS_RECORD_BYTES, dtype=torch.uint8, pin_memory=True)
        host.copy_(rec[:n * LAS_RECORD_BYTES])
        return host.numpy().reshape(n, LAS_RECORD_BYTES), list(offsets), mm.cpu().numpy()


def las_header(n: int, scale: float, offsets, int_minmax) -> bytes:
    """LAS 1.2 public header block (227 bytes, no VLRs) for point format 2, laspy's defaults."""
    today = datetime.date.today()
    mins = [int_minmax[k] * scale + offsets[k] for k in range(3)]
    maxs = [int_minmax[3 + k] * scale + offsets[k] for k in range(3)]
    h = struct.pack("<4sHH16sBB32s32sHHHIIBHI5I", b"LASF", 0, 0, b"\0" * 16, 1, 2,
                    b"OTHER".ljust(32, b"\0"), b"laspy".ljust(32, b"\0"),
                    today.timetuple().tm_yday, today.year, 227, 227, 0, 2, LAS_RECORD_BYTES, n, 0, 0, 0, 0, 0)
    h += struct.pack("<12d", scale, scale, scale, offsets[0], offsets[1], offsets[2],
                     maxs[0], mins[0], maxs[1], mins[1], maxs[2], mins[2])
    assert len(h) == 227
    return h


def save_las(points, colors, filename: str, device=None) -> str:
    """Save as LAS format for GIS compatibility (reference save_las, app.py:343-377)."""
    filepath = f"outputs/{filename}.las"
    scale = 0.01
    if points is None or len(points) == 0:
        raise ValueError("No points to write to LAS")
    rec, offsets, mm = las_point_records(points, colors, scale, None, device)
    with open(filepath, "wb") as f:
        f.write(las_header(len(rec), scale, offsets, mm))
        f.write(rec.tobytes())
    return filepath


# ---- PLY (Open3D write_point_cloud, app.py:329-341) -------------------------------------------
PLY_HEADER = ("ply\nformat binary_little_endian 1.0\ncomment Created by Open3D\nelement vertex {n}\n"
              "property double x\nproperty double y\nproperty double z\n"
              "property uchar red\nproperty uchar green\nproperty uchar blue\nend_header\n")
# Open3D's writer puts the normals after z when the cloud has them
PLY_NORMAL_HEADER = ("ply\nformat binary_little_endian 1.0\ncomment Created by Open3D\nelement vertex {n}\n"
                     "property double x\nproperty double y\nproperty double z\n"
                     "property double nx\nproperty double ny\nproperty double nz\n"
                     "property uchar red\nproperty uchar green\nproperty uchar blue\nend_header\n")


def _device_normals(normals, n: int, dev) -> torch.Tensor:
    if isinstance(normals, torch.Tensor):
        nrm = normals.to(dev)
    else:
        nrm = torch.from_numpy(np.ascontiguousarray(normals, dtype=np.float64)).to(dev)
    if nrm.dtype != torch.float64 or tuple(nrm.shape) != (n, 3):
        raise ValueError("normals must be float64 [N, 3] for N points")
    return nrm.contiguous()


def ply_vertex_records(points, colors, device=None, normals=None) -> np.ndarray:
    """-> uint8 [n, 27]: float64 x, y, z and uchar r, g, b per vertex; with ``normals`` (float64 [n, 3]) uint8
    [n, 51]: float64 x, y, z, nx, ny, nz and uchar r, g, b."""
    lib = _lib.load_library()
    xyz, rgb, count, n = _device_rows(points, colors, device)
    rb = PLY_RECORD_BYTES if normals is None else PLY_NORMAL_RECORD_BYTES
    if n == 0:
        return np.zeros((0, rb), np.uint8)
    dev = xyz.device
    with torch.cuda.device(dev):
        rec = torch.empty(n * rb + 16, dtype=torch.uint8, device=dev)
        if normals is None:
            check(lib.d2pc_ply_records_enqueue(xyz.data_ptr(), rgb.data_ptr(), count.data_ptr(), n, rec.data_ptr(),
                                               _stream(dev)), "d2pc_ply_records_enqueue")
        else:
            nrm = _device_normals(normals, n, dev)
            check(lib.d2pc_ply_normal_records_enqueue(xyz.data_ptr(), nrm.data_ptr(), rgb.data_ptr(), count.data_ptr(),
                                                      n, rec.data_ptr(), _stream(dev)), "d2pc_ply_normal_records_enqueue")
        host = torch.empty(n * rb, dtype=torch.uint8, pin_memory=True)
        host.copy_(rec[:n * rb])
        return host.numpy().reshape(n, rb)


def save_ply(points, colors, filename: str, device=None, normals=None) -> str:
    """Save as PLY format (reference save_ply, app.py:329-341); with ``normals`` the vertices carry nx, ny, nz."""
    filepath = f"outputs/{filename}.ply"
    rec = ply_vertex_records(points, colors, device, normals=normals)
    header = PLY_HEADER if normals is None else PLY_NORMAL_HEADER
    with open(filepath, "wb") as f:
        f.write(header.format(n=len(rec)).encode("ascii"))
        f.write(rec.tobytes())
    return filepath


# ---- mesh PLY (Open3D write_triangle_mesh, row m1) --------------------------------------------
# the vertex header of the point-cloud PLY plus Open3D's face element
PLY_FACE_ELEMENT = "element face {m}\nproperty list uchar uint vertex_indices\n"
PLY_MESH_HEADER = PLY_HEADER.replace("end_header\n", PLY_FACE_ELEMENT + "end_header\n")
PLY_MESH_NORMAL_HEADER = PLY_NORMAL_HEADER.replace("end_header\n", PLY_FACE_ELEMENT + "end_header\n")


def ply_face_records(triangles, device=None) -> np.ndarray:
    """-> uint8 [t, 13]: uchar 3 and the three vertex ids as uint32 per triangle (int32 [t, 3] in)."""
    lib = _lib.load_library()
    if isinstance(triangles, torch.Tensor):
        tri = triangles
    else:
        dev = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        tri = torch.from_numpy(np.ascontiguousarray(triangles, dtype=np.int32).reshape(-1, 3)).to(dev)
    if tri.dtype != torch.int32 or tri.dim() != 2 or tri.shape[1] != 3:
        raise ValueError("triangles must be int32 [T, 3]")
    t = int(tri.shape[0])
    if t == 0:
        return np.zeros((0, PLY_FACE_RECORD_BYTES), np.uint8)
    dev = tri.device
    with torch.cuda.device(dev):
        tri = tri.contiguous()
        cnt = torch.tensor([t], dtype=torch.int32, device=dev)
        rec = torch.empty(t * PLY_FACE_RECORD_BYTES + 16, dtype=torch.uint8, device=dev)
        check(lib.d2pc_ply_face_records_enqueue(tri.data_ptr(), cnt.data_ptr(), t, rec.data_ptr(), _stream(dev)),
              "d2pc_ply_face_records_enqueue")
        host = torch.empty(t * PLY_FACE_RECORD_BYTES, dtype=torch.uint8, pin_memory=True)
        host.copy_(rec[:t * PLY_FACE_RECORD_BYTES])
        return host.numpy().reshape(t, PLY_FACE_RECORD_BYTES)


def _mesh_ply_parts(mesh, device=None):
    """-> (header bytes, vertex records, face records) of a TriangleMesh (NumPy arrays or CUDA tensors)."""
    nrm = mesh.vertex_normals
    dev = mesh.vertices.device if isinstance(mesh.vertices, torch.Tensor) else device
    vrec = ply_vertex_records(mesh.vertices, mesh.colors, dev, normals=nrm)
    frec = ply_face_records(mesh.triangles, dev)
    header = PLY_MESH_HEADER if nrm is None else PLY_MESH_NORMAL_HEADER
    return header.format(n=len(vrec), m=len(frec)).encode("ascii"), vrec, frec


def mesh_ply_bytes(mesh, device=None) -> bytes:
    """The binary PLY Open3D's ``write_triangle_mesh`` writes for the mesh: vertices (float64 x, y, z, then nx, ny,
    nz when the mesh has normals, uchar red, green, blue) and 13-byte faces."""
    head, vrec, frec = _mesh_ply_parts(mesh, device)
    return head + vrec.tobytes() + frec.tobytes()


def save_mesh_ply(mesh, filename: str, device=None) -> str:
    """Write the mesh as ``outputs/<filename>.ply`` (``mesh_ply_bytes``) and return the path, like ``save_ply``."""
    filepath = f"outputs/{filename}.ply"
    head, vrec, frec = _mesh_ply_parts(mesh, device)
    Path("outputs").mkdir(exist_ok=True)
    with open(filepath, "wb") as f:
        f.write(head)
        f.write(vrec)   # straight from the pinned buffers (either may be empty)
        f.write(frec)
    return filepath


def save_point_cloud(points, colors, format: str, filename: str, device=None) -> str:
    """Save point cloud in various formats (reference save_point_cloud, app.py:310-327)."""
    try:
        Path("outputs").mkdir(exist_ok=True)
        if format.lower() == "ply":
            return save_ply(points, colors, filename, device)
        elif format.lower() in ["las", "laz"]:
            return save_las(points, colors, filename, device)
        elif format.lower() == "xyz":
            return save_xyz(points, colors, filename, device)
        else:
            raise ValueError(f"Unsupported format: {format}")
    except Exception as e:
        logger.error(f"Error saving point cloud: {str(e)}")
        raise
