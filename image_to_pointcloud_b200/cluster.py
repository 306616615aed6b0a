"""Row f5: density clustering of a point cloud on the GPU, Open3D's ``cluster_dbscan`` and ``remove_radius_outlier``
(spec: oracle/d2pc_cluster_oracle.py), run by ``d2pc_dbscan_enqueue`` / ``d2pc_radius_outlier_enqueue``.

Statistical outlier removal keeps a compact floater of twenty or more points, because each of its points has close
neighbours.  Clustering finds it: ``remove_small_clusters`` drops the noise and the clusters below ``min_size``
points.  ``points`` / ``colors`` may be NumPy arrays (uploaded once) or CUDA tensors; ``return_device=True`` leaves
the results on the device.  Every function reads back one small block (the kept count, the error word and the cluster
count) per call.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

from . import _lib
from ._lib import check
from .writers import _device_rows, _stream

GRID_CELL_LIMIT = 1048574.0    # cells per axis the device grid holds (d2pc_grid.cuh, kSorCellLimit)
RADIUS_MESSAGE = "Illegal input parameters, number of points and radius must be positive"


def check_eps(eps, name: str = "eps") -> float:
    e = float(eps)
    if not (math.isfinite(e) and e > 0.0 and 0.0 < e * e < math.inf):
        raise ValueError(f"{name} must be a finite positive number")
    return e


def check_min_points(min_points, name: str = "min_points") -> int:
    k = int(min_points)
    if k != min_points or k < 0 or k > 0x7FFFFFFF:
        raise ValueError(f"{name} must be an integer >= 0")
    return k


def check_min_size(min_size, name: str = "min_size") -> int:
    k = int(min_size)
    if k != min_size or k < 1 or k > 0xFFFFFFFF:
        raise ValueError(f"{name} must be an integer >= 1")
    return k


def _grid_message(eps: float) -> str:
    return (f"eps {eps!r} is too small for the extent of the cloud: the grid holds fewer than {int(GRID_CELL_LIMIT)} "
            f"cells of side eps / 2 per axis")


def _check_host_points(points, eps: float) -> None:
    """Host arrays are checked before any device work; device tensors by the kernels' error word."""
    if isinstance(points, torch.Tensor):
        return
    p = np.asarray(points, dtype=np.float32)
    if p.ndim != 2 or p.shape[1] != 3:
        raise ValueError("points must be float32 [N, 3]")
    if len(p) == 0:
        return
    if not np.isfinite(p).all():
        raise ValueError("points must be finite")
    lo, hi = p.min(axis=0).astype(np.float64), p.max(axis=0).astype(np.float64)
    cs = eps * 0.5 * (1.0 + 2.0 ** -20)
    if not all((h - l if h > l else 0.0) / cs < GRID_CELL_LIMIT for l, h in zip(lo, hi)):
        raise ValueError(_grid_message(eps))


def _raise_for(err: int, eps: float) -> None:
    if err & _lib.CLUSTER_ERR_NONFINITE:
        raise ValueError("points must be finite")
    if err & _lib.CLUSTER_ERR_GRID:
        raise ValueError(_grid_message(eps))
    if err:
        raise RuntimeError(f"density clustering failed on the device (error bits {err})")


def _run(points, colors, eps, *, min_points=None, min_size=None, nb_points=None, compact=True, device=None):
    """One call of the DBSCAN (nb_points None) or the radius-outlier kernels.  Returns a dict of device tensors:
    labels / sizes (DBSCAN), xyz / rgb / index (compact), and the host ints kept, clusters."""
    lib = _lib.load_library()
    has_colors = colors is not None and len(colors) == len(points)
    xyz, rgb, count, n = _device_rows(points, colors if has_colors else None, device)
    dev = xyz.device
    out = {"kept": 0, "clusters": 0}
    with torch.cuda.device(dev):
        if n == 0:
            out["labels"] = torch.zeros(0, dtype=torch.int32, device=dev)
            out["sizes"] = torch.zeros(0, dtype=torch.int32, device=dev)
            out["xyz"], out["rgb"], out["index"] = xyz, (rgb if has_colors else None), torch.zeros(0, dtype=torch.int32,
                                                                                                 device=dev)
            return out
        nb = C.c_size_t(0)
        check(lib.d2pc_cluster_scratch_bytes(n, C.byref(nb)), "d2pc_cluster_scratch_bytes")
        scratch = torch.empty(int(nb.value), dtype=torch.uint8, device=dev)
        keys = torch.empty(6, dtype=torch.int32, device=dev)
        bounds = torch.empty(6, dtype=torch.float32, device=dev)
        s = _stream(dev)
        check(lib.d2pc_rows_bounds_enqueue(xyz.data_ptr(), count.data_ptr(), n, keys.data_ptr(), bounds.data_ptr(), s),
              "d2pc_rows_bounds_enqueue")
        counts = torch.zeros(4, dtype=torch.int32, device=dev)
        oxyz = torch.empty_like(xyz) if compact else None
        orgb = torch.empty_like(rgb) if compact and has_colors else None
        oidx = torch.empty(n, dtype=torch.int32, device=dev) if compact else None
        ptr = (lambda t: t.data_ptr() if t is not None else None)
        if nb_points is None:
            labels = torch.empty(n, dtype=torch.int32, device=dev)
            sizes = torch.empty(n, dtype=torch.int32, device=dev)
            check(lib.d2pc_dbscan_enqueue(xyz.data_ptr(), rgb.data_ptr() if orgb is not None else None, count.data_ptr(),
                                          n, bounds.data_ptr(), eps, min_points, min_size if min_size else 1,
                                          scratch.data_ptr(), scratch.numel(), labels.data_ptr(), sizes.data_ptr(),
                                          ptr(oxyz), ptr(orgb), ptr(oidx), counts.data_ptr(), s), "d2pc_dbscan_enqueue")
        else:
            check(lib.d2pc_radius_outlier_enqueue(xyz.data_ptr(), rgb.data_ptr() if has_colors else None,
                                                  count.data_ptr(), n, bounds.data_ptr(), nb_points, eps,
                                                  scratch.data_ptr(), scratch.numel(), ptr(oxyz), ptr(orgb), ptr(oidx),
                                                  counts.data_ptr(), s), "d2pc_radius_outlier_enqueue")
        kept, err, clusters, _ = (int(v) for v in counts.cpu())
        _raise_for(err, eps)
        out.update(kept=kept, clusters=clusters)
        if nb_points is None:
            out["labels"], out["sizes"] = labels, sizes[:clusters]
        if compact:
            out["xyz"], out["rgb"], out["index"] = oxyz[:kept], (orgb[:kept] if orgb is not None else None), oidx[:kept]
        return out


def _rows(r, return_device: bool):
    if return_device:
        return r["xyz"], r["rgb"], r["index"]
    return (r["xyz"].cpu().numpy(), r["rgb"].cpu().numpy() if r["rgb"] is not None else None,
            r["index"].cpu().numpy().astype(np.int64))


def cluster_dbscan(points, eps: float, min_points: int, *, device=None, return_device: bool = False):
    """``np.asarray(pcd.cluster_dbscan(eps, min_points))``: int32 [N] cluster labels, -1 for noise.  Clusters are
    numbered by their lowest core point, as Open3D numbers them."""
    eps, min_points = check_eps(eps), check_min_points(min_points)
    _check_host_points(points, eps)
    r = _run(points, None, eps, min_points=min_points, compact=False, device=device)
    return r["labels"] if return_device else r["labels"].cpu().numpy()


def remove_radius_outlier(points, colors=None, *, nb_points: int, radius: float, device=None,
                          return_device: bool = False):
    """``pcd.remove_radius_outlier(nb_points, radius)``: the rows with more than ``nb_points`` neighbours within
    ``radius`` (the row itself counted), in input order -> (points, colors or None, kept_index)."""
    r = float(radius)
    k = int(nb_points)
    if k != nb_points or k < 1 or k > 0x7FFFFFFE or not (math.isfinite(r) and r > 0.0 and 0.0 < r * r < math.inf):
        raise ValueError(RADIUS_MESSAGE)
    _check_host_points(points, r)
    return _rows(_run(points, colors, r, nb_points=k, device=device), return_device)


def remove_small_clusters(points, colors=None, *, eps: float, min_points: int, min_size: int = 1, device=None,
                          return_device: bool = False):
    """The rows of the DBSCAN clusters (``cluster_dbscan(points, eps, min_points)``) of at least ``min_size`` points,
    in input order; noise is dropped -> (points, colors or None, kept_index)."""
    eps, min_points, min_size = check_eps(eps), check_min_points(min_points), check_min_size(min_size)
    _check_host_points(points, eps)
    return _rows(_run(points, colors, eps, min_points=min_points, min_size=min_size, device=device), return_device)
