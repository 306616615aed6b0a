"""Point normals on the device, with the semantics of Open3D's ``estimate_normals`` -- the first step of the
reference's mesh builder (backend/app.py:271-308) -- followed by ``orient_normals_towards_camera_location``:

    normals = estimate_normals(points)                      # float64 [N, 3], like np.asarray(pcd.normals)
    pcd.normals = o3d.utility.Vector3dVector(normals)

Run by ``d2pc_normals_enqueue``: exact k-nearest neighbours through the same uniform grid as the outlier removal
(float64 distances, ties ordered by (distance, row)), Open3D's covariance, its fast 3x3 eigen solver in float64.
``points`` may be a NumPy array (uploaded once) or a CUDA tensor.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import check
from .writers import _device_rows, _stream

MAX_KNN = 64


def estimate_normals(points, *, knn: int = 30, radius=None, orient_towards=(0.0, 0.0, 0.0),
                     return_covariances: bool = False, device=None, return_device: bool = False):
    """Normal of every point from its ``knn`` nearest points (itself included); with ``radius`` only the points
    closer than ``radius`` count (Open3D's ``KDTreeSearchParamHybrid(radius, knn)``).  Fewer than 3 neighbours give
    (0, 0, 1).  Normals are flipped to face ``orient_towards`` (default: the camera at the origin of the stage's
    frame); ``orient_towards=None`` keeps the solver's sign.

    Returns float64 [N, 3] normals, and with ``return_covariances`` also the float64 [N, 3, 3] covariances
    (Open3D's ``pcd.covariances``).  NumPy arrays, or CUDA tensors with ``return_device``."""
    knn = int(knn)
    if not 1 <= knn <= MAX_KNN:
        raise ValueError(f"knn must be in 1..{MAX_KNN}")
    r = 0.0 if radius is None else float(radius)
    if radius is not None and not (np.isfinite(r) and r > 0.0):
        raise ValueError("radius must be a positive finite number or None")
    cam = None
    if orient_towards is not None:
        cam = np.ascontiguousarray(orient_towards, dtype=np.float64).reshape(-1)
        if cam.shape != (3,) or not np.isfinite(cam).all():
            raise ValueError("orient_towards must be three finite numbers or None")
    lib = _lib.load_library()
    xyz, _, count, n = _device_rows(points, None, device)
    dev = xyz.device
    with torch.cuda.device(dev):
        normals = torch.empty((n, 3), dtype=torch.float64, device=dev)
        cov = torch.empty((n, 6), dtype=torch.float64, device=dev) if return_covariances else None
        if n > 0:
            if not bool(torch.isfinite(xyz).all()):
                raise ValueError("estimate_normals: non-finite coordinates")
            nb = C.c_size_t(0)
            check(lib.d2pc_normals_scratch_bytes(n, C.byref(nb)), "d2pc_normals_scratch_bytes")
            scratch = torch.empty(int(nb.value), dtype=torch.uint8, device=dev)
            keys = torch.empty(6, dtype=torch.int32, device=dev)
            bounds = torch.empty(6, dtype=torch.float32, device=dev)
            s = _stream(dev)
            check(lib.d2pc_rows_bounds_enqueue(xyz.data_ptr(), count.data_ptr(), n, keys.data_ptr(), bounds.data_ptr(), s),
                  "d2pc_rows_bounds_enqueue")
            cam_c = (C.c_double * 3)(*cam) if cam is not None else None
            check(lib.d2pc_normals_enqueue(xyz.data_ptr(), count.data_ptr(), n, bounds.data_ptr(), knn, r,
                                           1 if cam is not None else 0, cam_c, scratch.data_ptr(), scratch.numel(),
                                           normals.data_ptr(), cov.data_ptr() if cov is not None else None, s),
                  "d2pc_normals_enqueue")
        if cov is not None:
            cov = cov[:, [0, 1, 2, 1, 3, 4, 2, 4, 5]].reshape(n, 3, 3)
        if not return_device:
            normals = normals.cpu().numpy()
            cov = cov.cpu().numpy() if cov is not None else None
        return (normals, cov) if return_covariances else normals
