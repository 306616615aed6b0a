"""Drop-in for the reference's ``depth_to_point_cloud`` (reference backend/app.py:174-250).

    points, colors = depth_to_point_cloud(image, depth, density=..., invert=..., depth_scale=...,
                                          smooth=..., fov=...)

is what ``process_image_pipeline`` calls (backend/app.py:468-476).  Same positional signature,
same return value (two C-contiguous float32 [N,3] NumPy arrays on the host, row
``i = (v/step) * ceil(W/step) + (u/step)``), same error convention (exceptions; ``KeyError`` for an
unknown density).  Extensions are keyword-only and default to "off": ``z_range`` (depth-range mask
with ordered compaction), ``drop_nonfinite``, ``voxel_size`` (voxel-grid down-sampling).

All arithmetic runs in the sm_100a kernels of libd2pc.so.  There is no CPU path in this package.
"""
from __future__ import annotations

import logging
import threading
from typing import Dict, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _device
from .engine import DENSITY_STEP, MAX_SMOOTH_KSIZE, EmitResult, FrameEngine, smoothing_kernel

logger = logging.getLogger(__name__)

# One engine (workspace + pinned / device staging buffers) per geometry and device, shared by all callers.
# Threading contract: the cache is guarded by _CACHE_LOCK, and every engine carries its own lock that is held
# from staging the inputs until the results have left the device, so concurrent calls (a thread pool,
# ``run_in_executor``) on the same geometry serialise instead of overwriting each other's staged frame; calls
# on different geometries or devices run concurrently.
_ENGINES: Dict[tuple, "FrameEngine"] = {}
_STAGING: Dict[tuple, dict] = {}
_CACHE_LOCK = threading.Lock()


def _engine_for(img_h, img_w, img_c, dep_h, dep_w, device) -> FrameEngine:
    dev = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
    key = (str(dev), img_h, img_w, img_c, dep_h, dep_w)
    with _CACHE_LOCK:
        return _engine_locked(key, dev, img_h, img_w, img_c, dep_h, dep_w)


def _engine_locked(key, dev, img_h, img_w, img_c, dep_h, dep_w) -> FrameEngine:
    eng = _ENGINES.get(key)
    if eng is None:
        if len(_ENGINES) > 8:  # geometry changes per upload in the web app; keep the cache small
            # engines still in use by another thread stay alive through that thread's reference
            _ENGINES.clear()
            _STAGING.clear()
        eng = FrameEngine(img_h, img_w, dep_h, dep_w, batch=1, img_c=img_c, device=dev)
        eng._staging = None
        _ENGINES[key] = eng
        with torch.cuda.device(dev):
            eng._staging = _STAGING[key] = dict(
                lock=threading.Lock(),
                depth_pin=torch.empty((1, dep_h, dep_w), dtype=torch.float32, pin_memory=True),
                depth_dev=torch.empty((1, dep_h, dep_w), dtype=torch.float32, device=dev),
                bgr_pin=(torch.empty((1, img_h, img_w, img_c), dtype=torch.uint8, pin_memory=True)
                         if img_c >= 3 else None),
                bgr_dev=(torch.empty((1, img_h, img_w, img_c), dtype=torch.uint8, device=dev)
                         if img_c >= 3 else None),
                count_pin=torch.zeros(1, dtype=torch.int32, pin_memory=True),
            )
    return eng


def _image_channels(image: np.ndarray) -> int:
    # reference: colours come from image[v, u][:3] when ndim == 3 and shape[2] >= 3, else grey 128
    if image.ndim == 3 and image.shape[2] >= 3:
        if image.shape[2] not in (3, 4):
            raise ValueError("images with more than 4 channels are not supported")
        return int(image.shape[2])
    return 1


def check_depth_dtype(depth: np.ndarray, img_h: int, img_w: int) -> None:
    """The reference resizes the depth map in its own dtype (cv2.resize, app.py:188) and casts to float32
    afterwards (app.py:191).  float32 maps (what run_depth_model returns, app.py:116) are interpolated exactly
    as the reference does.  Any dtype is accepted when no resize is needed (the cast is then all that happens).
    A float64 map that needs a resize is cast to float32 FIRST and interpolated in float32: a documented
    deviation (the reference interpolates in float64 and casts afterwards; measured <= 7e-6 relative on the
    resized map, DESIGN.md section 7).  Integer maps that need a resize are refused: cv2 rounds the interpolated
    values back to integers (fixed-point / IPP integer arithmetic), which a float32 interpolation cannot
    reproduce within the 1e-5 tolerance."""
    if tuple(depth.shape[:2]) == (img_h, img_w) or depth.dtype in (np.float32, np.float64):
        return
    raise TypeError(f"depth of dtype {depth.dtype} needs a resize to {(img_h, img_w)}: pass float32 "
                    "(the reference's depth model output, app.py:116), float64, or a map of the image's size")


def depth_to_point_cloud(image: np.ndarray, depth: np.ndarray,
                         density: str = "medium",
                         invert: bool = True,
                         depth_scale: float = 10.0,
                         smooth: bool = False,
                         smooth_ksize: int = 5,
                         fov: Optional[float] = None,
                         *,
                         z_range: Optional[Tuple[float, float]] = None,
                         drop_nonfinite: bool = False,
                         voxel_size: Optional[float] = None,
                         return_voxel_index: bool = False,
                         return_bounds: bool = False,
                         pinned: bool = True,
                         device=None) -> tuple:
    """Convert a depth map to a coloured 3-D point cloud on a B200 (see module docstring).

    ``pinned=True`` (default) returns arrays backed by page-locked host memory (the device -> host copy runs at
    PCIe speed and the call returns as soon as it lands); a caller that keeps many results alive (the reference
    keeps each job's arrays, app.py:540-559) can pass ``pinned=False`` to get ordinary pageable arrays instead.
    Thread-safe: calls on the same geometry serialise on the engine's lock."""
    try:
        if not isinstance(image, np.ndarray) or not isinstance(depth, np.ndarray):
            raise TypeError("image and depth must be numpy arrays")
        img_h, img_w = image.shape[:2]
        dep_h, dep_w = depth.shape[:2]
        step = DENSITY_STEP[density]  # noqa: F841  (KeyError like the reference, before any work)
        if image.dtype != np.uint8:
            raise TypeError("image must be uint8 (cv2.imdecode output)")
        check_depth_dtype(depth, int(img_h), int(img_w))
        if smooth and len(smoothing_kernel(smooth_ksize)) > MAX_SMOOTH_KSIZE:
            # the reference accepts any size (cv2.GaussianBlur); this build keeps the coefficients in kernel
            # arguments and stops at 255 taps -- refused before any GPU work (the reference's only caller uses 5)
            raise ValueError(f"smooth_ksize {smooth_ksize} gives a kernel larger than {MAX_SMOOTH_KSIZE}")
        img_c = _image_channels(image)
        eng = _engine_for(int(img_h), int(img_w), img_c, int(dep_h), int(dep_w), device)
        st = eng._staging
        with st["lock"]:
            return _run_locked(eng, st, image, depth, img_c, dep_h, dep_w, density, invert, depth_scale, smooth,
                               smooth_ksize, fov, z_range, drop_nonfinite, voxel_size, return_voxel_index,
                               return_bounds, pinned)
    except Exception as e:  # same convention as the reference (app.py:248-250): log and re-raise
        logger.error(f"Error in point cloud generation: {str(e)}")
        raise


def _unpin(a: np.ndarray, pinned: bool) -> np.ndarray:
    return a if pinned else np.array(a, copy=True)


def _run_locked(eng, st, image, depth, img_c, dep_h, dep_w, density, invert, depth_scale, smooth, smooth_ksize, fov,
                z_range, drop_nonfinite, voxel_size, return_voxel_index, return_bounds, pinned):
    want_voxel = voxel_size is not None
    cfg = eng.make_config(density=density, invert=invert, depth_scale=float(depth_scale), fov=fov,
                          z_range=z_range, drop_nonfinite=drop_nonfinite,
                          want_bounds=(want_voxel or return_bounds))
    stream = torch.cuda.current_stream(eng.device)
    with torch.cuda.device(eng.device):
        # host -> pinned staging -> device (d = depth.astype(np.float32), app.py:191)
        st["depth_pin"][0].copy_(torch.from_numpy(np.ascontiguousarray(depth, dtype=np.float32).reshape(dep_h, dep_w)))
        st["depth_dev"].copy_(st["depth_pin"], non_blocking=True)
        if img_c >= 3:
            st["bgr_pin"][0].copy_(torch.from_numpy(np.ascontiguousarray(image)))
            st["bgr_dev"].copy_(st["bgr_pin"], non_blocking=True)
        # Without a mask every grid point is emitted: the row count is known, so the device -> host copies
        # are enqueued behind the emit and the call synchronises once.
        plain = z_range is None and not drop_nonfinite and not want_voxel
        host = {}

        def copy_out(xyz, rgb, count, bounds):
            for key, t in (("xyz", xyz), ("rgb", rgb)):
                if key not in host:
                    host[key] = torch.empty(t.shape[1:], dtype=t.dtype, pin_memory=True)
                host[key].copy_(t[0], non_blocking=True)
            if bounds is not None:
                if "bounds" not in host:
                    host["bounds"] = torch.empty((6,), dtype=torch.float32, pin_memory=True)
                host["bounds"].copy_(bounds[0], non_blocking=True)

        res = eng.process(cfg, st["depth_dev"], st["bgr_dev"], stream=stream,
                          smooth_ksize=(smooth_ksize if smooth else None), after_emit=copy_out if plain else None)
        if plain:   # process() has synchronised the stream
            out = (_unpin(host["xyz"].numpy(), pinned), _unpin(host["rgb"].numpy(), pinned))
            if return_bounds:
                out = out + (bounds_dict(host["bounds"].numpy()),)
            return out
        if want_voxel:
            vxyz, vrgb, vidx, vcount = eng.voxel_downsample(cfg, res, float(voxel_size),
                                                            want_index=return_voxel_index, stream=stream)
            n = int(vcount.cpu()[0])
            out = (_unpin(_device.pinned(vxyz[0, :n]), pinned), _unpin(_device.pinned(vrgb[0, :n]), pinned))
            if return_voxel_index:
                out = out + (vidx[0, :n].cpu().numpy(),)
            return out
        n = int(res.count.cpu()[0])
        out = (_unpin(_device.pinned(res.xyz[0, :n]), pinned), _unpin(_device.pinned(res.rgb[0, :n]), pinned))
        if return_bounds:
            out = out + (bounds_dict(res.bounds[0].cpu().numpy()),)
        return out


def _lattice_emit(image: np.ndarray, depth: np.ndarray, density: str, invert: bool, depth_scale: float, smooth: bool,
                  smooth_ksize: int, fov: Optional[float], device):
    """The unmasked emit of ``depth_to_point_cloud`` (same positional arguments) left on the device, for the stages
    that continue from it: -> (device, xyz, rgb, n), the ``n`` lattice rows in this call's own tensors.  The engine's
    lock is held while the engine runs; what the caller does with the rows does not need it."""
    img_h, img_w = image.shape[:2]
    dep_h, dep_w = depth.shape[:2]
    check_depth_dtype(depth, int(img_h), int(img_w))
    img_c = _image_channels(image)
    eng = _engine_for(int(img_h), int(img_w), img_c, int(dep_h), int(dep_w), device)
    dev = eng.device
    cfg = eng.make_config(density=density, invert=invert, depth_scale=float(depth_scale), fov=fov)
    n = eng.points_per_frame(cfg)   # the emit is unmasked: every lattice point is a row
    with eng._staging["lock"], torch.cuda.device(dev):
        d = torch.from_numpy(np.ascontiguousarray(depth, dtype=np.float32).reshape(1, dep_h, dep_w)).to(dev)
        im = torch.from_numpy(np.ascontiguousarray(image).reshape(1, img_h, img_w, -1)).to(dev) if img_c >= 3 else None
        res = eng.process(cfg, d, im, stream=torch.cuda.current_stream(dev),
                          smooth_ksize=(smooth_ksize if smooth else None))
    return dev, res.xyz[0, :n], res.rgb[0, :n], n


DEPTH_PREVIEW_MAX = 2048  # reference backend/app.py:44


def depth_preview_bgr(depth: np.ndarray, invert: bool = True, device=None) -> np.ndarray:
    """Device part of the reference's create_depth_preview (app.py:127-153): robust normalisation of
    the un-resized depth map, 8-bit quantisation and the PLASMA colour map.  uint8 [h, w, 3] BGR."""
    d = np.ascontiguousarray(depth, dtype=np.float32)
    h, w = d.shape[:2]
    eng = _engine_for(int(h), int(w), 1, int(h), int(w), device)
    with eng._staging["lock"], torch.cuda.device(eng.device):
        dev = torch.from_numpy(d.reshape(1, h, w)).to(eng.device)
        return eng.depth_preview(dev, invert=invert)[0].cpu().numpy()


def create_depth_preview(depth: np.ndarray, invert: bool = True, device=None) -> Optional[str]:
    """Drop-in for the reference's create_depth_preview (app.py:124-172): base64 PNG data URL of the
    colour-mapped depth map, or None on failure (logged), like the reference.  Normalisation and
    colour mapping run on the GPU; the optional INTER_AREA down-scale and the PNG encoder stay on the
    host (OpenCV), as in the reference."""
    try:
        import base64

        import cv2
        colored = depth_preview_bgr(depth, invert=invert, device=device)
        dh, dw = colored.shape[:2]
        dmax = max(dh, dw)
        if dmax > DEPTH_PREVIEW_MAX:
            s = DEPTH_PREVIEW_MAX / float(dmax)
            colored = cv2.resize(colored, (int(round(dw * s)), int(round(dh * s))), interpolation=cv2.INTER_AREA)
        ok, buf = cv2.imencode('.png', colored)
        if not ok:
            raise ValueError("Failed to encode depth image")
        return "data:image/png;base64," + base64.b64encode(buf.tobytes()).decode('utf-8')
    except Exception as e:
        logger.error(f"Failed to create depth preview: {e}")
        return None


def bounds_dict(b6: np.ndarray) -> dict:
    """The "bounds" block of the reference's GIS metadata (generate_gis_metadata, app.py:393-400;
    also the LAS offsets of save_las, app.py:352), from the min/max reduction fused into emit."""
    return {"minX": float(b6[0]), "maxX": float(b6[3]), "minY": float(b6[1]), "maxY": float(b6[4]),
            "minZ": float(b6[2]), "maxZ": float(b6[5])}


def depth_to_point_cloud_batch(images: Sequence[np.ndarray], depths: Sequence[np.ndarray],
                               density: str = "medium", invert: bool = True, depth_scale: float = 10.0,
                               fov: Optional[float] = None, *, z_range=None, drop_nonfinite: bool = False,
                               chunk: int = 8, device=None):
    """Many frames of one geometry through the same path: list of (points, colors) per frame.

    Host buffers in, host buffers out.  Frames are processed ``chunk`` at a time with three
    streams (H2D / kernels / D2H) and double-buffered pinned staging, so copies overlap compute.
    """
    from .hostpipe import HostFramePipeline
    if len(images) != len(depths):
        raise ValueError("images and depths differ in length")
    if len(images) == 0:
        return []
    img_h, img_w = images[0].shape[:2]
    dep_h, dep_w = depths[0].shape[:2]
    img_c = _image_channels(images[0])
    for d in depths:
        check_depth_dtype(d, int(img_h), int(img_w))
    pipe = HostFramePipeline(img_h, img_w, dep_h, dep_w, img_c=img_c, chunk=min(chunk, len(images)),
                             density=density, invert=invert, depth_scale=depth_scale, fov=fov,
                             z_range=z_range, drop_nonfinite=drop_nonfinite, device=device)
    return pipe.run(images, depths)
