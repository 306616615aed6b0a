"""Row m1: a triangle mesh of one frame on the device, from the image lattice its points come from.

The unmasked emit row ``i = r * C + c`` comes from pixel ``(r * step, c * step)`` of an ``R x C = ceil(H / step) x
ceil(W / step)`` lattice, so every point's neighbours are known without a search.  Each lattice quad is split into
two triangles along its shorter diagonal; triangles that are degenerate, face away from the camera, or are seen at
more than ``max_angle`` degrees from their normal (the ones that bridge a depth discontinuity) are dropped.  This is
the standard depth-image triangulation, not the reference's Poisson / BPA mesh builder (backend/app.py:271-308): it
runs in milliseconds and is deterministic, and the spec is our own (DESIGN.md, row m1).

    mesh = depth_to_mesh(image, depth, density="medium", z_range=(0.5, 9.5), refine=True)
    save_mesh_ply(mesh, "scene")                          # outputs/scene.ply, Open3D's binary layout

Run by ``d2pc_grid_mesh_enqueue``; vertex normals follow Open3D's ``ComputeVertexNormals`` (float64).
``simplify_mesh`` (row m2, ``d2pc_mesh_simplify_enqueue``) reduces such a mesh by vertex clustering, e.g. for a preview:

    small = simplify_mesh(mesh, voxel_size=0.02)           # contraction="average" or "quadric"

Row m3 (``d2pc_mesh_components_enqueue``, ``d2pc_mesh_filter_enqueue``) finds the edge-connected components of a
mesh (Open3D ``cluster_connected_triangles``) and removes triangles by a mask, e.g. the small islands a depth cut
leaves in front of the surface:

    clean = remove_small_components(mesh, min_triangles=10)

Row m4 (``d2pc_mesh_smooth_enqueue``, ``d2pc_mesh_vertex_normals_enqueue``) smooths a mesh (Open3D
``filter_smooth_simple`` / ``filter_smooth_laplacian`` / ``filter_smooth_taubin``) and recomputes the vertex normals of
any mesh, e.g. to take the terraces of a monocular depth map out of the lattice mesh:

    smooth = compute_vertex_normals(filter_smooth_taubin(mesh, 10, scope="vertex"))
"""
from __future__ import annotations

import ctypes as C
import math
from typing import NamedTuple, Optional

import numpy as np
import torch

from . import _lib
from ._lib import check
from .api import _engine_for, _image_channels, check_depth_dtype
from .engine import DENSITY_STEP
from .refine import statistical_outlier_removal
from .writers import _device_rows, _stream


class TriangleMesh(NamedTuple):
    vertices: object               # float32 [V, 3]
    colors: object                 # float32 [V, 3] (0..255, like the point cloud's colours)
    triangles: object              # int32 [T, 3] vertex ids, ordered by lattice quad
    vertex_normals: Optional[object]   # float64 [V, 3] or None
    vertex_rows: object            # int64 [V] lattice row of every vertex


def _cos2(max_angle) -> float:
    a = float(max_angle)
    if not 0.0 < a <= 90.0:
        raise ValueError("max_angle must be in (0, 90] degrees")
    c = math.cos(math.radians(a))
    return c * c


def _max_edge(max_edge) -> float:
    if max_edge is None:
        return 0.0
    e = float(max_edge)
    if not (np.isfinite(e) and e > 0.0):
        raise ValueError("max_edge must be a positive finite number or None")
    return e


def grid_mesh(points, colors, lattice_shape, *, keep=None, max_edge=None, max_angle: float = 85.0,
              remove_unreferenced: bool = True, compute_normals: bool = True, device=None,
              return_device: bool = False) -> TriangleMesh:
    """Triangle mesh of the ``lattice_shape = (R, C)`` lattice rows ``points`` / ``colors`` (float32 [R*C, 3]).

    A row is a vertex only when ``keep`` (bool / uint8 [R*C], optional) holds and its coordinates are finite; with
    ``remove_unreferenced`` only rows used by a kept triangle stay.  ``max_edge`` drops triangles with a longer edge,
    ``max_angle`` (degrees, (0, 90]) those seen at a more grazing angle.  NumPy arrays, or CUDA tensors with
    ``return_device``."""
    R, Cc = int(lattice_shape[0]), int(lattice_shape[1])
    if R < 1 or Cc < 1 or R * Cc >= 2 ** 31:
        raise ValueError("lattice_shape must be (R, C) with R, C >= 1 and R * C < 2^31")
    cos2, me = _cos2(max_angle), _max_edge(max_edge)
    lib = _lib.load_library()
    xyz, rgb, _, n = _device_rows(points, colors, device)
    if n != R * Cc:
        raise ValueError(f"{n} rows do not form a {R} x {Cc} lattice")
    dev = xyz.device
    with torch.cuda.device(dev):
        keep_t = None
        if keep is not None:
            keep_t = keep if isinstance(keep, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(keep))
            keep_t = keep_t.to(dev).reshape(-1)
            if keep_t.numel() != n:
                raise ValueError("keep must have one entry per lattice row")
            keep_t = (keep_t != 0).to(torch.uint8).contiguous()
        nb = C.c_size_t(0)
        check(lib.d2pc_grid_mesh_scratch_bytes(R, Cc, C.byref(nb)), "d2pc_grid_mesh_scratch_bytes")
        scratch = torch.empty(int(nb.value), dtype=torch.uint8, device=dev)
        vxyz = torch.empty((n, 3), dtype=torch.float32, device=dev)
        vrgb = torch.empty((n, 3), dtype=torch.float32, device=dev)
        vrow = torch.empty(n, dtype=torch.int32, device=dev)
        vnrm = torch.empty((n, 3), dtype=torch.float64, device=dev) if compute_normals else None
        tri = torch.empty((max(2 * (R - 1) * (Cc - 1), 1), 3), dtype=torch.int32, device=dev)
        counts = torch.zeros(2, dtype=torch.int32, device=dev)   # vertices, triangles
        flags = (_lib.MESH_REMOVE_UNREFERENCED if remove_unreferenced else 0) | \
            (_lib.MESH_NORMALS if compute_normals else 0)
        check(lib.d2pc_grid_mesh_enqueue(xyz.data_ptr(), rgb.data_ptr(), keep_t.data_ptr() if keep_t is not None else None,
                                         R, Cc, me, cos2, flags, scratch.data_ptr(), scratch.numel(), vxyz.data_ptr(),
                                         vrgb.data_ptr(), vrow.data_ptr(), vnrm.data_ptr() if vnrm is not None else None,
                                         counts.data_ptr(), tri.data_ptr(), counts.data_ptr() + 4, _stream(dev)),
              "d2pc_grid_mesh_enqueue")
        nv, nt = (int(v) for v in counts.cpu())
        mesh = TriangleMesh(vxyz[:nv], vrgb[:nv], tri[:nt], vnrm[:nv] if vnrm is not None else None,
                            vrow[:nv].to(torch.int64))
        if return_device:
            return mesh
        return TriangleMesh(*(t.cpu().numpy() if t is not None else None for t in mesh))


CONTRACTIONS = ("average", "quadric")
_SIMPLIFY_ERRORS = ((1, "voxel_size is too small."), (2, "a triangle refers to a vertex that does not exist"),
                    (4, "the mesh has a non-finite vertex (coordinate, colour or normal)"))


def check_voxel_size(voxel_size) -> float:
    vs = float(voxel_size)
    if not (math.isfinite(vs) and vs > 0.0):
        raise ValueError("voxel_size must be a positive finite number")
    return vs


def _device_array(x, dtype, cols, dev):
    if isinstance(x, torch.Tensor):
        t = x.to(dev)
    else:
        np_dtype = {torch.float32: np.float32, torch.float64: np.float64, torch.int32: np.int32, torch.int64: np.int64}
        t = torch.from_numpy(np.ascontiguousarray(x, dtype=np_dtype[dtype])).to(dev)
    if t.dtype != dtype:
        raise ValueError(f"expected {dtype}, got {t.dtype}")
    return (t.reshape(-1, cols) if cols else t.reshape(-1)).contiguous()


def simplify_mesh(mesh: TriangleMesh, voxel_size: float, *, contraction: str = "average", device=None,
                  return_device: bool = False) -> TriangleMesh:
    """Row m2: vertex-clustering simplification (Open3D ``simplify_vertex_clustering``) of a ``TriangleMesh`` -- the
    NumPy arrays ``grid_mesh`` returns or its CUDA tensors.  Every occupied voxel of size ``voxel_size`` (the ax-2
    grid on the vertices' bounds) becomes one vertex, ordered by its lowest member vertex; ``contraction`` places it
    at the members' mean ("average") or at the minimiser of their triangles' plane quadrics when that is well
    conditioned and inside the voxel ("quadric").  Colours are averaged and normals (when the mesh has them) summed
    and normalised; triangles are remapped, collapsed and repeated ones dropped.  Raises ValueError for bad
    arguments, a voxel index of 2^21 or more, a triangle id outside the vertices, and a non-finite vertex."""
    vs = check_voxel_size(voxel_size)
    if contraction not in CONTRACTIONS:
        raise ValueError(f"contraction must be one of {CONTRACTIONS}")
    nv, nt = len(mesh.vertices), len(mesh.triangles)
    if nv >= 2 ** 24 or nt >= 2 ** 31:
        raise ValueError("simplify_mesh takes fewer than 2^24 vertices and 2^31 triangles")
    lib = _lib.load_library()
    if not torch.cuda.is_available():
        raise RuntimeError("image_to_pointcloud_b200 needs a CUDA device (no CPU fallback exists)")
    if isinstance(mesh.vertices, torch.Tensor):
        dev = mesh.vertices.device
    else:
        dev = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
    with torch.cuda.device(dev):
        xyz = _device_array(mesh.vertices, torch.float32, 3, dev)
        rgb = _device_array(mesh.colors, torch.float32, 3, dev)
        tri = _device_array(mesh.triangles, torch.int32, 3, dev)
        rows = _device_array(mesh.vertex_rows, torch.int64, 0, dev)
        nrm = None if mesh.vertex_normals is None else _device_array(mesh.vertex_normals, torch.float64, 3, dev)
        if len(rgb) != nv or len(rows) != nv or (nrm is not None and len(nrm) != nv):
            raise ValueError("colors, vertex_rows and vertex_normals must have one row per vertex")
        nb = C.c_size_t(0)
        check(lib.d2pc_mesh_simplify_scratch_bytes(nv, nt, C.byref(nb)), "d2pc_mesh_simplify_scratch_bytes")
        scratch = torch.empty(int(nb.value), dtype=torch.uint8, device=dev)
        oxyz = torch.empty((nv, 3), dtype=torch.float32, device=dev)
        orgb = torch.empty((nv, 3), dtype=torch.float32, device=dev)
        orow = torch.empty(nv, dtype=torch.int64, device=dev)
        onrm = torch.empty((nv, 3), dtype=torch.float64, device=dev) if nrm is not None else None
        otri = torch.empty((nt, 3), dtype=torch.int32, device=dev)
        words = torch.zeros(3, dtype=torch.int32, device=dev)   # vertices, triangles, error
        flags = (_lib.SIMPLIFY_QUADRIC if contraction == "quadric" else 0) | (_lib.SIMPLIFY_NORMALS if nrm is not None else 0)

        def ptr(t):
            return t.data_ptr() if t is not None and t.numel() > 0 else None
        check(lib.d2pc_mesh_simplify_enqueue(ptr(xyz), ptr(rgb), ptr(nrm), ptr(rows), nv, ptr(tri), nt, vs, flags,
                                             scratch.data_ptr(), scratch.numel(), ptr(oxyz), ptr(orgb), ptr(onrm),
                                             ptr(orow), words.data_ptr(), ptr(otri), words.data_ptr() + 4,
                                             words.data_ptr() + 8, _stream(dev)),
              "d2pc_mesh_simplify_enqueue")
        kv, kt, err = (int(v) for v in words.cpu())
        if err:
            raise ValueError("; ".join(msg for bit, msg in _SIMPLIFY_ERRORS if err & bit))
        out = TriangleMesh(oxyz[:kv], orgb[:kv], otri[:kt], onrm[:kv] if onrm is not None else None, orow[:kv])
        if return_device:
            return out
        return TriangleMesh(*(t.cpu().numpy() if t is not None else None for t in out))


_COMPONENT_ERRORS = ((1, "a triangle refers to a vertex that does not exist"),
                     (2, "the mesh has a non-finite vertex coordinate"))
_COMPONENT_MAX_TRIANGLES = 2 ** 25


def _mesh_device(mesh, device):
    lib = _lib.load_library()
    if not torch.cuda.is_available():
        raise RuntimeError("image_to_pointcloud_b200 needs a CUDA device (no CPU fallback exists)")
    if len(mesh.triangles) > _COMPONENT_MAX_TRIANGLES or len(mesh.vertices) > 2 ** 31:
        raise ValueError("meshes of at most 2^25 triangles and 2^31 vertices are supported")
    if isinstance(mesh.vertices, torch.Tensor):
        return lib, mesh.vertices.device
    return lib, torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")


def _raise_component_errors(err: int, where: str) -> None:
    if err & ~3:
        raise RuntimeError(f"{where}: a device loop exhausted its bound (error word {err})")
    if err:
        raise ValueError("; ".join(msg for bit, msg in _COMPONENT_ERRORS if err & bit))


def _ptr(t):
    return t.data_ptr() if t is not None and t.numel() > 0 else None


def cluster_connected_triangles(mesh: TriangleMesh, *, device=None, return_device: bool = False):
    """Row m3: Open3D's ``cluster_connected_triangles`` of a ``TriangleMesh`` (NumPy arrays or CUDA tensors):
    ``(triangle_clusters int32 [T], cluster_n_triangles int64 [K], cluster_area float64 [K])``.  Two triangles are
    connected when they share an edge; clusters are numbered by their lowest triangle.  Areas are Open3D's triangle
    areas summed in 64-bit fixed point (DESIGN.md, row m3), so they repeat bit for bit.  Raises ValueError for a
    triangle id outside the vertices and a non-finite vertex coordinate."""
    lib, dev = _mesh_device(mesh, device)
    nv, nt = len(mesh.vertices), len(mesh.triangles)
    with torch.cuda.device(dev):
        xyz = _device_array(mesh.vertices, torch.float32, 3, dev)
        tri = _device_array(mesh.triangles, torch.int32, 3, dev)
        nb = C.c_size_t(0)
        check(lib.d2pc_mesh_components_scratch_bytes(nv, nt, C.byref(nb)), "d2pc_mesh_components_scratch_bytes")
        scratch = torch.empty(int(nb.value), dtype=torch.uint8, device=dev)
        labels = torch.empty(nt, dtype=torch.int32, device=dev)
        n = torch.empty(nt, dtype=torch.int64, device=dev)
        area = torch.empty(nt, dtype=torch.float64, device=dev)
        words = torch.zeros(2, dtype=torch.int32, device=dev)   # K, error
        check(lib.d2pc_mesh_components_enqueue(_ptr(xyz), nv, _ptr(tri), nt, scratch.data_ptr(), scratch.numel(),
                                               _ptr(labels), _ptr(n), _ptr(area), words.data_ptr(),
                                               words.data_ptr() + 4, _stream(dev)),
              "d2pc_mesh_components_enqueue")
        k, err = (int(v) for v in words.cpu())
        _raise_component_errors(err, "cluster_connected_triangles")
        out = (labels, n[:k], area[:k])
        if return_device:
            return out
        return tuple(t.cpu().numpy() for t in out)


def remove_triangles_by_mask(mesh: TriangleMesh, mask, *, remove_unreferenced: bool = True, device=None,
                             return_device: bool = False) -> TriangleMesh:
    """Row m3: Open3D's ``remove_triangles_by_mask`` (``mask`` bool [T], True: the triangle goes), then with
    ``remove_unreferenced`` its ``remove_unreferenced_vertices``.  Kept triangles and vertices keep their order;
    colours, normals and vertex rows are carried unchanged (normals are not recomputed).  Raises ValueError for a
    triangle id outside the vertices and a non-finite vertex coordinate."""
    lib, dev = _mesh_device(mesh, device)
    nv, nt = len(mesh.vertices), len(mesh.triangles)
    with torch.cuda.device(dev):
        m = mask if isinstance(mask, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(mask))
        m = m.to(dev).reshape(-1)
        if m.numel() != nt:
            raise ValueError("the mask must have one entry per triangle")
        keep = (m == 0).to(torch.uint8).contiguous()
        return _filter(lib, dev, mesh, keep, remove_unreferenced, return_device)


def _filter(lib, dev, mesh, keep, remove_unreferenced, return_device):
    nv, nt = len(mesh.vertices), len(mesh.triangles)
    xyz = _device_array(mesh.vertices, torch.float32, 3, dev)
    rgb = _device_array(mesh.colors, torch.float32, 3, dev)
    tri = _device_array(mesh.triangles, torch.int32, 3, dev)
    rows = _device_array(mesh.vertex_rows, torch.int64, 0, dev)
    nrm = None if mesh.vertex_normals is None else _device_array(mesh.vertex_normals, torch.float64, 3, dev)
    if len(rgb) != nv or len(rows) != nv or (nrm is not None and len(nrm) != nv):
        raise ValueError("colors, vertex_rows and vertex_normals must have one row per vertex")
    nb = C.c_size_t(0)
    check(lib.d2pc_mesh_filter_scratch_bytes(nv, nt, C.byref(nb)), "d2pc_mesh_filter_scratch_bytes")
    scratch = torch.empty(int(nb.value), dtype=torch.uint8, device=dev)
    oxyz = torch.empty((nv, 3), dtype=torch.float32, device=dev)
    orgb = torch.empty((nv, 3), dtype=torch.float32, device=dev)
    orow = torch.empty(nv, dtype=torch.int64, device=dev)
    onrm = torch.empty((nv, 3), dtype=torch.float64, device=dev) if nrm is not None else None
    otri = torch.empty((nt, 3), dtype=torch.int32, device=dev)
    words = torch.zeros(3, dtype=torch.int32, device=dev)   # vertices, triangles, error
    flags = (_lib.MESH_REMOVE_UNREFERENCED if remove_unreferenced else 0) | (_lib.MESH_NORMALS if nrm is not None else 0)
    check(lib.d2pc_mesh_filter_enqueue(_ptr(xyz), _ptr(rgb), _ptr(nrm), _ptr(rows), nv, _ptr(tri), nt, _ptr(keep),
                                       flags, scratch.data_ptr(), scratch.numel(), _ptr(oxyz), _ptr(orgb), _ptr(onrm),
                                       _ptr(orow), words.data_ptr(), _ptr(otri), words.data_ptr() + 4,
                                       words.data_ptr() + 8, _stream(dev)),
          "d2pc_mesh_filter_enqueue")
    kv, kt, err = (int(v) for v in words.cpu())
    _raise_component_errors(err, "remove_triangles_by_mask")
    out = TriangleMesh(oxyz[:kv], orgb[:kv], otri[:kt], onrm[:kv] if onrm is not None else None, orow[:kv])
    if return_device:
        return out
    return TriangleMesh(*(t.cpu().numpy() if t is not None else None for t in out))


def check_min_triangles(min_triangles) -> int:
    n = int(min_triangles)
    if n != min_triangles or n < 1:
        raise ValueError("min_triangles must be an integer >= 1")
    return n


def _small_components(mesh, min_triangles, min_area, remove_unreferenced, device, return_device):
    """(cleaned mesh, K, removed triangles)."""
    if min_triangles is None and min_area is None:
        raise ValueError("give min_triangles, min_area or both")
    if min_triangles is not None:
        min_triangles = check_min_triangles(min_triangles)
    if min_area is not None:
        min_area = float(min_area)
        if math.isnan(min_area):
            raise ValueError("min_area must be a number")
    lib, dev = _mesh_device(mesh, device)
    with torch.cuda.device(dev):
        labels, n, area = cluster_connected_triangles(mesh, device=dev, return_device=True)
        lab = labels.to(torch.int64)
        remove = torch.zeros(labels.numel(), dtype=torch.bool, device=dev)
        if min_triangles is not None:
            remove |= n[lab] < min_triangles
        if min_area is not None:
            remove |= area[lab] < min_area
        keep = (~remove).to(torch.uint8)
        out = _filter(lib, dev, mesh, keep, remove_unreferenced, return_device)
        return out, int(n.numel()), len(mesh.triangles) - len(out.triangles)


def remove_small_components(mesh: TriangleMesh, *, min_triangles: Optional[int] = None,
                            min_area: Optional[float] = None, device=None, return_device: bool = False) -> TriangleMesh:
    """Row m3: removes every connected component (``cluster_connected_triangles``) with fewer than ``min_triangles``
    triangles or less area than ``min_area``, then the vertices no kept triangle uses -- Open3D's
    ``remove_triangles_by_mask(cluster_n_triangles[triangle_clusters] < N)`` and ``remove_unreferenced_vertices``,
    entirely on the device.  Raises ValueError for bad arguments, a triangle id outside the vertices and a non-finite
    vertex coordinate."""
    return _small_components(mesh, min_triangles, min_area, True, device, return_device)[0]


SMOOTH_SCOPES = {"all": _lib.SMOOTH_VERTEX | _lib.SMOOTH_NORMAL | _lib.SMOOTH_COLOR, "vertex": _lib.SMOOTH_VERTEX,
                 "normal": _lib.SMOOTH_NORMAL, "color": _lib.SMOOTH_COLOR}
_SMOOTH_ERRORS = ((1, "a triangle refers to a vertex that does not exist"),
                  (2, "the mesh has a non-finite vertex coordinate (or colour / normal in the scope)"))


def check_iterations(number_of_iterations) -> int:
    n = int(number_of_iterations)
    if n != number_of_iterations or not 0 <= n < 2 ** 31:
        raise ValueError("number_of_iterations must be an integer >= 0")
    return n


def _finite(name, x) -> float:
    x = float(x)
    if not math.isfinite(x):
        raise ValueError(f"{name} must be a finite number")
    return x


def _host_or_device(out, return_device):
    if return_device:
        return out
    return TriangleMesh(*(t.cpu().numpy() if t is not None else None for t in out))


def _smooth(mesh, method, iterations, lambda_filter, mu, scope, device, return_device):
    n = check_iterations(iterations)
    lam, mu = _finite("lambda_filter", lambda_filter), _finite("mu", mu)
    if scope not in SMOOTH_SCOPES:
        raise ValueError(f"scope must be one of {tuple(SMOOTH_SCOPES)}")
    lib, dev = _mesh_device(mesh, device)
    nv, nt = len(mesh.vertices), len(mesh.triangles)
    with torch.cuda.device(dev):
        xyz = _device_array(mesh.vertices, torch.float32, 3, dev)
        rgb = _device_array(mesh.colors, torch.float32, 3, dev)
        tri = _device_array(mesh.triangles, torch.int32, 3, dev)
        rows = _device_array(mesh.vertex_rows, torch.int64, 0, dev)
        nrm = None if mesh.vertex_normals is None else _device_array(mesh.vertex_normals, torch.float64, 3, dev)
        if len(rgb) != nv or len(rows) != nv or (nrm is not None and len(nrm) != nv):
            raise ValueError("colors, vertex_rows and vertex_normals must have one row per vertex")
        nb = C.c_size_t(0)
        check(lib.d2pc_mesh_smooth_scratch_bytes(nv, nt, C.byref(nb)), "d2pc_mesh_smooth_scratch_bytes")
        scratch = torch.empty(int(nb.value), dtype=torch.uint8, device=dev)
        oxyz = torch.empty((nv, 3), dtype=torch.float32, device=dev)
        orgb = torch.empty((nv, 3), dtype=torch.float32, device=dev)
        onrm = torch.empty((nv, 3), dtype=torch.float64, device=dev) if nrm is not None else None
        err = torch.zeros(1, dtype=torch.int32, device=dev)
        check(lib.d2pc_mesh_smooth_enqueue(_ptr(xyz), _ptr(rgb), _ptr(nrm), nv, _ptr(tri), nt, method, n, lam, mu,
                                           SMOOTH_SCOPES[scope], scratch.data_ptr(), scratch.numel(), _ptr(oxyz),
                                           _ptr(orgb), _ptr(onrm), err.data_ptr(), _stream(dev)),
              "d2pc_mesh_smooth_enqueue")
        e = int(err.cpu())
        _raise_smooth_errors(e, "mesh smoothing")
        return _host_or_device(TriangleMesh(oxyz, orgb, tri, onrm, rows), return_device)


def _raise_smooth_errors(err: int, where: str) -> None:
    if err & ~3:
        raise RuntimeError(f"{where}: a device loop exhausted its bound (error word {err})")
    if err:
        raise ValueError("; ".join(msg for bit, msg in _SMOOTH_ERRORS if err & bit))


def filter_smooth_simple(mesh: TriangleMesh, number_of_iterations: int = 1, *, scope: str = "all", device=None,
                         return_device: bool = False) -> TriangleMesh:
    """Row m4: Open3D's ``filter_smooth_simple`` of a ``TriangleMesh`` (NumPy arrays or CUDA tensors): every pass
    moves each vertex to the mean of itself and its neighbours (Open3D's adjacency sets, visited in ascending id),
    in float64, rounded to float32 once at the end.  ``scope`` ("all", "vertex", "normal", "color") picks the fields
    filtered (normals only when the mesh has them; they are not renormalised); triangles and vertex rows are kept.
    Raises ValueError for bad arguments, a triangle id outside the vertices and a non-finite value."""
    return _smooth(mesh, _lib.SMOOTH_SIMPLE, number_of_iterations, 0.5, -0.53, scope, device, return_device)


def filter_smooth_laplacian(mesh: TriangleMesh, number_of_iterations: int = 1, lambda_filter: float = 0.5, *,
                            scope: str = "all", device=None, return_device: bool = False) -> TriangleMesh:
    """Row m4: Open3D's ``filter_smooth_laplacian``: every pass moves each vertex by ``lambda_filter`` towards the mean
    of its neighbours weighted by 1 / (distance + 1e-12); colours and normals take the same weights.  A vertex
    without neighbours stays as it is (Open3D writes NaN).  Otherwise as ``filter_smooth_simple``."""
    return _smooth(mesh, _lib.SMOOTH_LAPLACIAN, number_of_iterations, lambda_filter, -0.53, scope, device,
                   return_device)


def filter_smooth_taubin(mesh: TriangleMesh, number_of_iterations: int = 1, lambda_filter: float = 0.5,
                         mu: float = -0.53, *, scope: str = "all", device=None,
                         return_device: bool = False) -> TriangleMesh:
    """Row m4: Open3D's ``filter_smooth_taubin``: every iteration is a Laplacian pass with ``lambda_filter``, then one
    with ``mu``, which smooths without the shrinking of the plain Laplacian.  Otherwise as
    ``filter_smooth_laplacian``."""
    return _smooth(mesh, _lib.SMOOTH_TAUBIN, number_of_iterations, lambda_filter, mu, scope, device, return_device)


def compute_vertex_normals(mesh: TriangleMesh, *, device=None, return_device: bool = False) -> TriangleMesh:
    """Row m4: the mesh with its ``vertex_normals`` replaced by Open3D's ``compute_vertex_normals``, m1's rule: the
    unnormalised normals of every vertex's triangles summed in ascending triangle order and normalised ((0, 0, 1) for
    a zero sum), float64 -- bit for bit the normals ``grid_mesh`` computes.  Raises ValueError for a triangle id
    outside the vertices and a non-finite vertex coordinate."""
    lib, dev = _mesh_device(mesh, device)
    nv, nt = len(mesh.vertices), len(mesh.triangles)
    with torch.cuda.device(dev):
        xyz = _device_array(mesh.vertices, torch.float32, 3, dev)
        rgb = _device_array(mesh.colors, torch.float32, 3, dev)
        tri = _device_array(mesh.triangles, torch.int32, 3, dev)
        rows = _device_array(mesh.vertex_rows, torch.int64, 0, dev)
        if len(rgb) != nv or len(rows) != nv:
            raise ValueError("colors and vertex_rows must have one row per vertex")
        nb = C.c_size_t(0)
        check(lib.d2pc_mesh_vertex_normals_scratch_bytes(nv, nt, C.byref(nb)), "d2pc_mesh_vertex_normals_scratch_bytes")
        scratch = torch.empty(int(nb.value), dtype=torch.uint8, device=dev)
        onrm = torch.empty((nv, 3), dtype=torch.float64, device=dev)
        err = torch.zeros(1, dtype=torch.int32, device=dev)
        check(lib.d2pc_mesh_vertex_normals_enqueue(_ptr(xyz), nv, _ptr(tri), nt, scratch.data_ptr(), scratch.numel(),
                                                   _ptr(onrm), err.data_ptr(), _stream(dev)),
              "d2pc_mesh_vertex_normals_enqueue")
        _raise_smooth_errors(int(err.cpu()), "compute_vertex_normals")
        return _host_or_device(TriangleMesh(xyz, rgb, tri, onrm, rows), return_device)


def lattice_shape(img_h: int, img_w: int, density: str):
    """(R, C) of the emit lattice: ceil(H / step) x ceil(W / step)."""
    s = DENSITY_STEP[density]
    return -(-int(img_h) // s), -(-int(img_w) // s)


def refined_keep(xyz: torch.Tensor, keep: Optional[torch.Tensor], nb_neighbors: int, std_ratio: float) -> torch.Tensor:
    """Statistical outlier removal on the kept lattice rows (all rows when ``keep`` is None), its kept index scattered
    back into a uint8 lattice mask: the rows ``refine_point_cloud`` keeps of the same cloud."""
    n = int(xyz.shape[0])
    rows = torch.arange(n, device=xyz.device) if keep is None else torch.nonzero(keep).reshape(-1)
    out = torch.zeros(n, dtype=torch.uint8, device=xyz.device)
    if rows.numel() > 0:
        _, _, idx, _ = statistical_outlier_removal(xyz[rows].contiguous(), None, nb_neighbors, std_ratio,
                                                   return_device=True)
        out[rows[idx.to(torch.int64)]] = 1
    return out


def depth_to_mesh(image: np.ndarray, depth: np.ndarray, density: str = "medium", invert: bool = True,
                  depth_scale: float = 10.0, smooth: bool = False, smooth_ksize: int = 5, fov: Optional[float] = None,
                  *, z_range=None, refine: bool = False, nb_neighbors: int = 20, std_ratio: float = 2.0,
                  max_edge=None, max_angle: float = 85.0, remove_unreferenced: bool = True,
                  compute_normals: bool = True, min_component_triangles: Optional[int] = None, device=None,
                  return_device: bool = False) -> TriangleMesh:
    """Mesh of one (image, depth) pair in one device-resident pass: the unmasked emit of ``depth_to_point_cloud``
    (same positional arguments), ``z_range`` as a mask on the lattice (the float32 rule of the depth-range mask),
    with ``refine`` statistical outlier removal of the remaining rows (``nb_neighbors``, ``std_ratio``), then
    ``grid_mesh``.  The vertices are the points ``depth_to_point_cloud(..., z_range=z_range)`` followed by
    ``refine_point_cloud`` would keep (those a kept triangle uses, with ``remove_unreferenced``).  With
    ``min_component_triangles`` the components of fewer triangles are removed (``remove_small_components``)."""
    DENSITY_STEP[density]  # KeyError first, like the reference
    if z_range is not None and len(z_range) != 2:
        raise ValueError("z_range must be (z_min, z_max)")
    _cos2(max_angle), _max_edge(max_edge)   # argument errors before any device work
    if min_component_triangles is not None:
        check_min_triangles(min_component_triangles)
    img_h, img_w = image.shape[:2]
    dep_h, dep_w = depth.shape[:2]
    check_depth_dtype(depth, int(img_h), int(img_w))
    img_c = _image_channels(image)
    eng = _engine_for(int(img_h), int(img_w), img_c, int(dep_h), int(dep_w), device)
    dev = eng.device
    cfg = eng.make_config(density=density, invert=invert, depth_scale=float(depth_scale), fov=fov)
    with eng._staging["lock"], torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev)
        d = torch.from_numpy(np.ascontiguousarray(depth, dtype=np.float32).reshape(1, dep_h, dep_w)).to(dev)
        im = torch.from_numpy(np.ascontiguousarray(image).reshape(1, img_h, img_w, -1)).to(dev) if img_c >= 3 else None
        res = eng.process(cfg, d, im, stream=stream, smooth_ksize=(smooth_ksize if smooth else None))
        n = eng.points_per_frame(cfg)
        xyz, rgb = res.xyz[0, :n], res.rgb[0, :n]
        keep = None
        if z_range is not None:   # z32 >= f32(z_min) and z32 <= f32(z_max)
            z = xyz[:, 2]
            keep = ((z >= float(np.float32(z_range[0]))) & (z <= float(np.float32(z_range[1])))).to(torch.uint8)
        if refine:
            keep = refined_keep(xyz, keep, nb_neighbors, std_ratio)
        if min_component_triangles is None:
            return grid_mesh(xyz, rgb, lattice_shape(img_h, img_w, density), keep=keep, max_edge=max_edge,
                             max_angle=max_angle, remove_unreferenced=remove_unreferenced,
                             compute_normals=compute_normals, return_device=return_device)
        mesh = grid_mesh(xyz, rgb, lattice_shape(img_h, img_w, density), keep=keep, max_edge=max_edge,
                         max_angle=max_angle, remove_unreferenced=remove_unreferenced,
                         compute_normals=compute_normals, return_device=True)
        return _small_components(mesh, min_component_triangles, None, remove_unreferenced, dev, return_device)[0]
