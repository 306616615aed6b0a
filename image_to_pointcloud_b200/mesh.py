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

import math
from typing import NamedTuple, Optional

import numpy as np
import torch

from . import _lib
from ._device import device_for, device_rows, ptr, raise_errors, scratch, stream, to_host, upload
from ._lib import check
from .api import _lattice_emit
from .engine import DENSITY_STEP
from .refine import statistical_outlier_removal


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
    xyz, rgb, _, n = device_rows(points, colors, device)
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
        buf = scratch(lib.d2pc_grid_mesh_scratch_bytes, R, Cc, dev=dev)
        vxyz = torch.empty((n, 3), dtype=torch.float32, device=dev)
        vrgb = torch.empty((n, 3), dtype=torch.float32, device=dev)
        vrow = torch.empty(n, dtype=torch.int32, device=dev)
        vnrm = torch.empty((n, 3), dtype=torch.float64, device=dev) if compute_normals else None
        tri = torch.empty((max(2 * (R - 1) * (Cc - 1), 1), 3), dtype=torch.int32, device=dev)
        counts = torch.zeros(2, dtype=torch.int32, device=dev)   # vertices, triangles
        flags = (_lib.MESH_REMOVE_UNREFERENCED if remove_unreferenced else 0) | \
            (_lib.MESH_NORMALS if compute_normals else 0)
        check(lib.d2pc_grid_mesh_enqueue(xyz.data_ptr(), rgb.data_ptr(), ptr(keep_t), R, Cc, me, cos2, flags,
                                         buf.data_ptr(), buf.numel(), vxyz.data_ptr(), vrgb.data_ptr(), vrow.data_ptr(),
                                         ptr(vnrm), counts.data_ptr(), tri.data_ptr(), counts.data_ptr() + 4,
                                         stream(dev)), "d2pc_grid_mesh_enqueue")
        nv, nt = (int(v) for v in counts.cpu())
        mesh = TriangleMesh(vxyz[:nv], vrgb[:nv], tri[:nt], vnrm[:nv] if vnrm is not None else None,
                            vrow[:nv].to(torch.int64))
        return to_host(mesh, return_device)


CONTRACTIONS = ("average", "quadric")
_SIMPLIFY_ERRORS = ((1, "voxel_size is too small."), (2, "a triangle refers to a vertex that does not exist"),
                    (4, "the mesh has a non-finite vertex (coordinate, colour or normal)"))


def check_voxel_size(voxel_size) -> float:
    vs = float(voxel_size)
    if not (math.isfinite(vs) and vs > 0.0):
        raise ValueError("voxel_size must be a positive finite number")
    return vs


def _mesh_inputs(mesh: TriangleMesh, dev, normals: bool = True):
    """-> (xyz, rgb, triangles, vertex rows, normals or None) of ``mesh`` on ``dev``; with ``normals=False`` the mesh's
    normals are left out."""
    nv = len(mesh.vertices)
    xyz = upload(mesh.vertices, torch.float32, 3, dev)
    rgb = upload(mesh.colors, torch.float32, 3, dev)
    tri = upload(mesh.triangles, torch.int32, 3, dev)
    rows = upload(mesh.vertex_rows, torch.int64, 0, dev)
    nrm = None if mesh.vertex_normals is None or not normals else upload(mesh.vertex_normals, torch.float64, 3, dev)
    if len(rgb) != nv or len(rows) != nv or (nrm is not None and len(nrm) != nv):
        raise ValueError("colors, vertex_rows and vertex_normals must have one row per vertex" if normals else
                         "colors and vertex_rows must have one row per vertex")
    return xyz, rgb, tri, rows, nrm


def _reduce_mesh(scratch_bytes, enqueue, mesh: TriangleMesh, arg, flags: int, errors, where: str, dev,
                 return_device: bool) -> TriangleMesh:
    """One call of ``d2pc_mesh_simplify_enqueue`` or ``d2pc_mesh_filter_enqueue``: the same inputs, outputs (at most
    the input's vertices and triangles) and word block (vertices, triangles, error) around an argument of their own,
    ``arg`` (the voxel size, the keep mask)."""
    nv, nt = len(mesh.vertices), len(mesh.triangles)
    xyz, rgb, tri, rows, nrm = _mesh_inputs(mesh, dev)
    buf = scratch(scratch_bytes, nv, nt, dev=dev)
    oxyz = torch.empty((nv, 3), dtype=torch.float32, device=dev)
    orgb = torch.empty((nv, 3), dtype=torch.float32, device=dev)
    orow = torch.empty(nv, dtype=torch.int64, device=dev)
    onrm = torch.empty((nv, 3), dtype=torch.float64, device=dev) if nrm is not None else None
    otri = torch.empty((nt, 3), dtype=torch.int32, device=dev)
    words = torch.zeros(3, dtype=torch.int32, device=dev)   # vertices, triangles, error
    check(enqueue(ptr(xyz), ptr(rgb), ptr(nrm), ptr(rows), nv, ptr(tri), nt, arg, flags, buf.data_ptr(), buf.numel(),
                  ptr(oxyz), ptr(orgb), ptr(onrm), ptr(orow), words.data_ptr(), ptr(otri), words.data_ptr() + 4,
                  words.data_ptr() + 8, stream(dev)), enqueue.__name__)
    kv, kt, err = (int(v) for v in words.cpu())
    raise_errors(err, errors, where)
    return to_host(TriangleMesh(oxyz[:kv], orgb[:kv], otri[:kt], onrm[:kv] if onrm is not None else None, orow[:kv]),
                   return_device)


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
    dev = device_for(mesh.vertices, device)
    flags = (_lib.SIMPLIFY_QUADRIC if contraction == "quadric" else 0) | \
        (_lib.SIMPLIFY_NORMALS if mesh.vertex_normals is not None else 0)
    with torch.cuda.device(dev):
        return _reduce_mesh(lib.d2pc_mesh_simplify_scratch_bytes, lib.d2pc_mesh_simplify_enqueue, mesh, vs, flags,
                            _SIMPLIFY_ERRORS, "simplify_mesh", dev, return_device)


_COMPONENT_ERRORS = ((1, "a triangle refers to a vertex that does not exist"),
                     (2, "the mesh has a non-finite vertex coordinate"))
_COMPONENT_MAX_TRIANGLES = 2 ** 25


def _mesh_device(mesh, device):
    lib, dev = _lib.load_library(), device_for(mesh.vertices, device)
    if len(mesh.triangles) > _COMPONENT_MAX_TRIANGLES or len(mesh.vertices) > 2 ** 31:
        raise ValueError("meshes of at most 2^25 triangles and 2^31 vertices are supported")
    return lib, dev


def cluster_connected_triangles(mesh: TriangleMesh, *, device=None, return_device: bool = False):
    """Row m3: Open3D's ``cluster_connected_triangles`` of a ``TriangleMesh`` (NumPy arrays or CUDA tensors):
    ``(triangle_clusters int32 [T], cluster_n_triangles int64 [K], cluster_area float64 [K])``.  Two triangles are
    connected when they share an edge; clusters are numbered by their lowest triangle.  Areas are Open3D's triangle
    areas summed in 64-bit fixed point (DESIGN.md, row m3), so they repeat bit for bit.  Raises ValueError for a
    triangle id outside the vertices and a non-finite vertex coordinate."""
    lib, dev = _mesh_device(mesh, device)
    nv, nt = len(mesh.vertices), len(mesh.triangles)
    with torch.cuda.device(dev):
        xyz = upload(mesh.vertices, torch.float32, 3, dev)
        tri = upload(mesh.triangles, torch.int32, 3, dev)
        buf = scratch(lib.d2pc_mesh_components_scratch_bytes, nv, nt, dev=dev)
        labels = torch.empty(nt, dtype=torch.int32, device=dev)
        n = torch.empty(nt, dtype=torch.int64, device=dev)
        area = torch.empty(nt, dtype=torch.float64, device=dev)
        words = torch.zeros(2, dtype=torch.int32, device=dev)   # K, error
        check(lib.d2pc_mesh_components_enqueue(ptr(xyz), nv, ptr(tri), nt, buf.data_ptr(), buf.numel(), ptr(labels),
                                               ptr(n), ptr(area), words.data_ptr(), words.data_ptr() + 4, stream(dev)),
              "d2pc_mesh_components_enqueue")
        k, err = (int(v) for v in words.cpu())
        raise_errors(err, _COMPONENT_ERRORS, "cluster_connected_triangles")
        return to_host((labels, n[:k], area[:k]), return_device)


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
    flags = (_lib.MESH_REMOVE_UNREFERENCED if remove_unreferenced else 0) | \
        (_lib.MESH_NORMALS if mesh.vertex_normals is not None else 0)
    return _reduce_mesh(lib.d2pc_mesh_filter_scratch_bytes, lib.d2pc_mesh_filter_enqueue, mesh, ptr(keep), flags,
                        _COMPONENT_ERRORS, "remove_triangles_by_mask", dev, return_device)


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


def _smooth(mesh, method, iterations, lambda_filter, mu, scope, device, return_device):
    n = check_iterations(iterations)
    lam, mu = _finite("lambda_filter", lambda_filter), _finite("mu", mu)
    if scope not in SMOOTH_SCOPES:
        raise ValueError(f"scope must be one of {tuple(SMOOTH_SCOPES)}")
    lib, dev = _mesh_device(mesh, device)
    nv, nt = len(mesh.vertices), len(mesh.triangles)
    with torch.cuda.device(dev):
        xyz, rgb, tri, rows, nrm = _mesh_inputs(mesh, dev)
        buf = scratch(lib.d2pc_mesh_smooth_scratch_bytes, nv, nt, dev=dev)
        oxyz = torch.empty((nv, 3), dtype=torch.float32, device=dev)
        orgb = torch.empty((nv, 3), dtype=torch.float32, device=dev)
        onrm = torch.empty((nv, 3), dtype=torch.float64, device=dev) if nrm is not None else None
        err = torch.zeros(1, dtype=torch.int32, device=dev)
        check(lib.d2pc_mesh_smooth_enqueue(ptr(xyz), ptr(rgb), ptr(nrm), nv, ptr(tri), nt, method, n, lam, mu,
                                           SMOOTH_SCOPES[scope], buf.data_ptr(), buf.numel(), ptr(oxyz), ptr(orgb),
                                           ptr(onrm), err.data_ptr(), stream(dev)), "d2pc_mesh_smooth_enqueue")
        raise_errors(int(err.cpu()), _SMOOTH_ERRORS, "mesh smoothing")
        return to_host(TriangleMesh(oxyz, orgb, tri, onrm, rows), return_device)


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
        xyz, rgb, tri, rows, _ = _mesh_inputs(mesh, dev, normals=False)
        buf = scratch(lib.d2pc_mesh_vertex_normals_scratch_bytes, nv, nt, dev=dev)
        onrm = torch.empty((nv, 3), dtype=torch.float64, device=dev)
        err = torch.zeros(1, dtype=torch.int32, device=dev)
        check(lib.d2pc_mesh_vertex_normals_enqueue(ptr(xyz), nv, ptr(tri), nt, buf.data_ptr(), buf.numel(), ptr(onrm),
                                                   err.data_ptr(), stream(dev)), "d2pc_mesh_vertex_normals_enqueue")
        raise_errors(int(err.cpu()), _SMOOTH_ERRORS, "compute_vertex_normals")
        return to_host(TriangleMesh(xyz, rgb, tri, onrm, rows), return_device)


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
    dev, xyz, rgb, _ = _lattice_emit(image, depth, density, invert, depth_scale, smooth, smooth_ksize, fov, device)
    img_h, img_w = image.shape[:2]
    with torch.cuda.device(dev):
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
