"""Row f1: drop-in for the reference's ``refine_point_cloud`` (backend/app.py:252-269): statistical outlier
removal with Open3D's semantics (``remove_statistical_outlier(nb_neighbors=20, std_ratio=2.0)``), run on
the GPU by ``d2pc_sor_enqueue`` (exact k-nearest neighbours through a uniform grid, float64 distances).

Same signature, return value and error convention as the reference: ``(points_f, colors_f)``; an empty or
``None`` cloud is returned as is; any failure is logged as a warning and the input is returned unchanged
(app.py:266-269).  ``points`` / ``colors`` may be NumPy arrays (uploaded once) or CUDA tensors.
"""
from __future__ import annotations

import logging

import numpy as np
import torch

from . import _lib
from ._device import device_rows, row_bounds, scratch, stream, to_host
from ._lib import check

logger = logging.getLogger(__name__)


def statistical_outlier_removal(points, colors=None, nb_neighbors: int = 20, std_ratio: float = 2.0, device=None,
                                return_device: bool = False):
    """-> (points_f, colors_f or None, kept_index, stats) with stats = dict(cloud_mean, std_dev, threshold)."""
    lib = _lib.load_library()
    has_colors = colors is not None and len(colors) == len(points)
    xyz, rgb, count, n = device_rows(points, colors if has_colors else None, device)
    dev = xyz.device
    with torch.cuda.device(dev):
        buf = scratch(lib.d2pc_sor_scratch_bytes, n, dev=dev)
        bounds = row_bounds(xyz, count, n, dev)
        oxyz = torch.empty_like(xyz)
        orgb = torch.empty_like(rgb) if has_colors else None
        oidx = torch.empty(n, dtype=torch.int32, device=dev)
        ocnt = torch.zeros(1, dtype=torch.int32, device=dev)
        stats = torch.zeros(4, dtype=torch.float64, device=dev)
        check(lib.d2pc_sor_enqueue(xyz.data_ptr(), rgb.data_ptr() if has_colors else None, count.data_ptr(), n,
                                   bounds.data_ptr(), int(nb_neighbors), float(std_ratio), buf.data_ptr(), buf.numel(),
                                   oxyz.data_ptr(), orgb.data_ptr() if has_colors else None, oidx.data_ptr(),
                                   ocnt.data_ptr(), stats.data_ptr(), stream(dev)), "d2pc_sor_enqueue")
        m = int(ocnt.cpu()[0])
        st = stats.cpu().numpy()
        info = {"cloud_mean": float(st[0]), "std_dev": float(st[1]), "threshold": float(st[2])}
        pts, cols, idx = to_host((oxyz[:m], orgb[:m] if has_colors else None, oidx[:m]), return_device)
        return pts, cols, (idx if return_device else idx.astype(np.int64)), info


def refine_point_cloud(points, colors, nb_neighbors: int = 20, std_ratio: float = 2.0) -> tuple:
    """Denoise point cloud using statistical outlier removal (reference app.py:252-269)."""
    try:
        if points is None or len(points) == 0:
            return points, colors
        if nb_neighbors < 1 or std_ratio <= 0:
            raise ValueError("Illegal input parameters, the number of neighbors and standard deviation ratio must be positive.")
        p, c, _, _ = statistical_outlier_removal(points, colors, nb_neighbors, std_ratio)
        return p, (c if c is not None else colors)
    except Exception as e:
        logger.warning(f"Point cloud refinement failed: {e}")
        return points, colors
