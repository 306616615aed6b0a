"""FrameEngine -- host side of the B200 depth-map -> point-cloud stage.

Owns the device workspace for one geometry (image size, depth size, batch) on one GPU and drives
the C-ABI library (include/d2pc.h) on a CUDA stream.  PyTorch is used only as the container for
device / pinned memory and for streams; every computation happens in libd2pc.so.  There is no CPU
or eager fallback: constructing an engine without a CUDA device or without the library raises.

A *frame* is one (image, depth) pair; a call processes ``batch`` frames that share geometry and
knobs.  Frames are independent (the reference function is pure, backend/app.py:174-250), which is
also how work is sharded across GPUs (see ``shard_frames``).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import D2pcConfig, D2pcFrameParams, check

DENSITY_STEP = {"low": 4, "medium": 2, "high": 1}  # reference backend/app.py:226


def reference_intrinsics(img_w: int, img_h: int, fov: Optional[float]) -> Tuple[float, float, float]:
    """cx, cy, f exactly as the reference computes them (backend/app.py:219-223)."""
    cx, cy = img_w / 2.0, img_h / 2.0
    if fov and fov > 0:
        f = (img_w / 2.0) / np.tan(np.deg2rad(fov) / 2.0)
    else:
        f = max(img_w, img_h) * 1.2
    return float(cx), float(cy), float(f)


_SMALL_GAUSSIAN = {  # cv2.getGaussianKernel(k, 0, CV_64F): fixed tables for k <= 9 (sigma <= 0)
    3: [0.25, 0.5, 0.25],
    5: [0.0625, 0.25, 0.375, 0.25, 0.0625],
    7: [0.03125, 0.109375, 0.21875, 0.28125, 0.21875, 0.109375, 0.03125],
    9: [4 / 256, 13 / 256, 30 / 256, 51 / 256, 60 / 256, 51 / 256, 30 / 256, 13 / 256, 4 / 256],
}
MAX_SMOOTH_KSIZE = 255


def smoothing_kernel(smooth_ksize) -> list:
    """k = max(3, int(smooth_ksize) // 2 * 2 + 1) (reference app.py:210) and the coefficients
    cv2.GaussianBlur(d, (k, k), 0) uses: OpenCV's fixed tables up to k = 9, else
    sigma = 0.15 k + 0.35, exp(-x^2 / (2 sigma^2)) normalised (OpenCV's getGaussianKernelBitExact)."""
    import math
    k = max(3, int(smooth_ksize) // 2 * 2 + 1)
    if k in _SMALL_GAUSSIAN:
        return list(_SMALL_GAUSSIAN[k])
    sigma = k * 0.15 + 0.35
    scale2x = -0.125 / (sigma * sigma)
    vals = [math.exp(float((2 * i - (k - 1)) ** 2) * scale2x) for i in range((k - 1) // 2)]
    total = 0.0
    for v in vals:
        total += v
    mul1 = 1.0 / (total * 2.0 + 1.0)
    half = [v * mul1 for v in vals]
    return half + [mul1] + half[::-1]


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


@dataclass
class EmitResult:
    xyz: torch.Tensor      # float32 [batch, N, 3] (device); rows [0, count[b]) valid per frame
    rgb: torch.Tensor      # float32 [batch, N, 3]
    count: torch.Tensor    # int32   [batch]
    bounds: Optional[torch.Tensor]  # float32 [batch, 6] or None


class FrameEngine:
    def __init__(self, img_h: int, img_w: int, dep_h: Optional[int] = None, dep_w: Optional[int] = None,
                 *, batch: int = 1, img_c: int = 3, device=None):
        if not torch.cuda.is_available():
            raise RuntimeError("image_to_pointcloud_b200 needs a CUDA device (no CPU fallback exists)")
        self.lib = _lib.load_library()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        if self.device.type != "cuda":
            raise RuntimeError("FrameEngine device must be a CUDA device")
        self.img_h, self.img_w, self.img_c = int(img_h), int(img_w), int(img_c)
        self.dep_h = int(dep_h if dep_h is not None else img_h)
        self.dep_w = int(dep_w if dep_w is not None else img_w)
        self.batch = int(batch)
        # workspace sized for the densest configuration (step 1) of this geometry
        cfg = self.make_config(density="high")
        nbytes = C.c_size_t(0)
        check(self.lib.d2pc_workspace_bytes(C.byref(cfg), C.byref(nbytes)), "d2pc_workspace_bytes")
        self.workspace_bytes = int(nbytes.value)
        with torch.cuda.device(self.device):
            self.workspace = torch.empty(self.workspace_bytes, dtype=torch.uint8, device=self.device)
            self._status = torch.zeros(self.batch, dtype=torch.int32, device=self.device)
            self._any = torch.zeros(1, dtype=torch.int32, device=self.device)
            self._any_host = torch.zeros(1, dtype=torch.int32, pin_memory=True)
        assert self.workspace.data_ptr() % 256 == 0
        self._voxel_table = None
        self._voxel_rows = None   # rows per frame the voxel table was last initialised for
        self._smooth_scratch = None
        self._path = None

    # ---- configuration -------------------------------------------------------------------
    def make_config(self, density: str = "high", invert: bool = True, depth_scale: float = 10.0,
                    fov: Optional[float] = None, z_range: Optional[Tuple[float, float]] = None,
                    drop_nonfinite: bool = False, want_bounds: bool = False,
                    force_fallback: bool = False) -> D2pcConfig:
        step = DENSITY_STEP[density]  # KeyError for unknown densities, like the reference
        cx, cy, f = reference_intrinsics(self.img_w, self.img_h, fov)
        cfg = D2pcConfig()
        cfg.batch = self.batch
        cfg.img_h, cfg.img_w, cfg.img_c = self.img_h, self.img_w, self.img_c
        cfg.dep_h, cfg.dep_w = self.dep_h, self.dep_w
        cfg.step = step
        cfg.invert = 1 if invert else 0
        cfg.depth_scale = float(depth_scale)
        cfg.cx, cfg.cy, cfg.f = cx, cy, f
        if z_range is not None:
            cfg.use_z_range = 1
            cfg.z_min, cfg.z_max = float(np.float32(z_range[0])), float(np.float32(z_range[1]))
        cfg.drop_nonfinite = 1 if drop_nonfinite else 0
        cfg.want_bounds = 1 if want_bounds else 0
        cfg.force_fallback = 1 if force_fallback else 0
        return cfg

    def points_per_frame(self, cfg: D2pcConfig) -> int:
        s = cfg.step
        return (-(-self.img_h // s)) * (-(-self.img_w // s))

    def alloc_outputs(self, cfg: D2pcConfig):
        n = self.points_per_frame(cfg)
        with torch.cuda.device(self.device):
            xyz = torch.empty((self.batch, n, 3), dtype=torch.float32, device=self.device)
            rgb = torch.empty((self.batch, n, 3), dtype=torch.float32, device=self.device)
        return xyz, rgb

    # ---- checks --------------------------------------------------------------------------
    def _check_inputs(self, depth: torch.Tensor, bgr: Optional[torch.Tensor]):
        if depth.device != self.device or depth.dtype != torch.float32 or not depth.is_contiguous():
            raise ValueError("depth must be a contiguous float32 tensor on the engine's device")
        if tuple(depth.shape) != (self.batch, self.dep_h, self.dep_w):
            raise ValueError(f"depth shape {tuple(depth.shape)} != {(self.batch, self.dep_h, self.dep_w)}")
        if self.img_c >= 3:
            if bgr is None or bgr.device != self.device or bgr.dtype != torch.uint8 or not bgr.is_contiguous():
                raise ValueError("bgr must be a contiguous uint8 tensor on the engine's device")
            if tuple(bgr.shape) != (self.batch, self.img_h, self.img_w, self.img_c):
                raise ValueError(f"bgr shape {tuple(bgr.shape)} != {(self.batch, self.img_h, self.img_w, self.img_c)}")

    def _stream(self, stream) -> int:
        s = stream if stream is not None else torch.cuda.current_stream(self.device)
        return s.cuda_stream

    def _call(self, name: str, *args) -> None:
        """One C-ABI call with the engine's device current (the library launches on the current device and
        sets kernel attributes there), whatever device the caller's thread has selected."""
        with torch.cuda.device(self.device):
            check(getattr(self.lib, name)(*args), name)

    # ---- asynchronous pieces (enqueue only, no host sync) ---------------------------------
    def enqueue_stats(self, cfg: D2pcConfig, depth: torch.Tensor, stream=None) -> None:
        self._call("d2pc_stats_enqueue", C.byref(cfg), depth.data_ptr(), self.workspace.data_ptr(),
                   self.workspace_bytes, self._stream(stream))

    def enqueue_stats_fallback(self, cfg: D2pcConfig, depth: torch.Tensor, stream=None) -> None:
        self._call("d2pc_stats_fallback_enqueue", C.byref(cfg), depth.data_ptr(), self.workspace.data_ptr(),
                   self.workspace_bytes, self._stream(stream))

    def enqueue_status(self, cfg: D2pcConfig, stream=None) -> None:
        """status words -> self._status, any-fallback flag -> pinned host word (async copy)."""
        self._call("d2pc_frame_status", C.byref(cfg), self.workspace.data_ptr(), self._status.data_ptr(),
                   self._any.data_ptr(), self._stream(stream))
        self._copy_flag(stream)

    def _copy_flag(self, stream=None) -> None:
        s = stream if stream is not None else torch.cuda.current_stream(self.device)
        with torch.cuda.device(self.device), torch.cuda.stream(s):
            self._any_host.copy_(self._any, non_blocking=True)

    def enqueue_emit(self, cfg: D2pcConfig, depth: torch.Tensor, bgr: Optional[torch.Tensor],
                     xyz: torch.Tensor, rgb: torch.Tensor, count: torch.Tensor,
                     bounds: Optional[torch.Tensor] = None, stream=None) -> None:
        self._call("d2pc_emit_enqueue", C.byref(cfg), depth.data_ptr(), _ptr(bgr), self.workspace.data_ptr(),
                   self.workspace_bytes, xyz.data_ptr(), rgb.data_ptr(), count.data_ptr(), _ptr(bounds),
                   self._stream(stream))

    # ---- the whole path as one sub-batch pipeline (csrc/d2pc_path.cu) -----------------------
    def enqueue_path(self, cfg: D2pcConfig, depth: torch.Tensor, bgr: Optional[torch.Tensor],
                     xyz: torch.Tensor, rgb: torch.Tensor, count: torch.Tensor,
                     bounds: Optional[torch.Tensor] = None, stream=None, *, sub_batch: Optional[int] = None,
                     lookahead: int = 0, graph: bool = False, flags: int = 0) -> None:
        """statistics + status + emit of the batch in ONE library call.  The per-frame status words land in
        ``self._status`` and the any-fallback flag in the pinned ``self._any_host`` (valid after the stream has
        been synchronised), like ``enqueue_status``.  ``graph=True`` replays a cached CUDA graph while the
        arguments repeat (steady-state batches on the same buffers).  ``sub_batch`` < batch pipelines the work
        over sub-batches on auxiliary streams, ``flags=PATH_ORDERED`` runs the index-ordered single-launch
        kernel: both bit-identical, both measured slower than one stage on B200 (kept for measurement)."""
        if self._path is None:
            h = C.c_void_p()
            self._call("d2pc_path_create", C.byref(h))
            self._path = h
        if sub_batch is None:
            sub_batch = self.default_sub_batch()
        self._call("d2pc_path_enqueue", self._path, C.byref(cfg), depth.data_ptr(), _ptr(bgr),
                   self.workspace.data_ptr(), self.workspace_bytes, xyz.data_ptr(), rgb.data_ptr(), count.data_ptr(),
                   _ptr(bounds), self._status.data_ptr(), self._any.data_ptr(), int(sub_batch), int(lookahead),
                   int(flags) | (_lib.PATH_GRAPH if graph else 0), self._stream(stream))
        self._copy_flag(stream)

    def default_sub_batch(self) -> int:
        """Frames per pipeline stage of ``enqueue_path``.  One stage (statistics of the whole batch, then its
        emit) is the fastest arrangement measured on B200: the emit is bound by DRAM writes at ~1.04 of the
        measured copy bandwidth, so statistics that run next to it only take bandwidth from it, and the L2 hit
        on the depth map saves less than the sub-batch overheads cost (DESIGN.md section 5)."""
        return self.batch

    def __del__(self):
        try:
            if getattr(self, "_path", None) is not None:
                with torch.cuda.device(self.device):
                    self.lib.d2pc_path_destroy(self._path)
                self._path = None
        except Exception:
            pass

    def enqueue_emit_smooth(self, cfg: D2pcConfig, smooth_ksize, depth: torch.Tensor,
                            bgr: Optional[torch.Tensor], xyz: torch.Tensor, rgb: torch.Tensor,
                            count: torch.Tensor, bounds: Optional[torch.Tensor] = None, stream=None) -> None:
        """a6: emission with cv2.GaussianBlur-compatible smoothing of the normalised map."""
        coeffs = smoothing_kernel(smooth_ksize)
        if len(coeffs) > MAX_SMOOTH_KSIZE:
            raise ValueError(f"smooth_ksize too large (kernel {len(coeffs)} > {MAX_SMOOTH_KSIZE})")
        nbytes = C.c_size_t(0)
        check(self.lib.d2pc_smooth_scratch_bytes(C.byref(cfg), C.byref(nbytes)), "d2pc_smooth_scratch_bytes")
        with torch.cuda.device(self.device):
            if self._smooth_scratch is None or self._smooth_scratch.numel() < nbytes.value:
                self._smooth_scratch = torch.empty(int(nbytes.value), dtype=torch.uint8, device=self.device)
        arr = (C.c_double * len(coeffs))(*coeffs)
        self._call("d2pc_emit_smooth_enqueue", C.byref(cfg), depth.data_ptr(), _ptr(bgr), self.workspace.data_ptr(),
                   self.workspace_bytes, len(coeffs), arr, self._smooth_scratch.data_ptr(),
                   self._smooth_scratch.numel(), xyz.data_ptr(), rgb.data_ptr(), count.data_ptr(), _ptr(bounds),
                   self._stream(stream))

    # ---- f2 depth preview ----------------------------------------------------------------
    def depth_preview(self, depth: torch.Tensor, invert: bool = True, stream=None) -> torch.Tensor:
        """Colour-mapped preview of every frame (reference create_depth_preview, app.py:127-153):
        uint8 [batch, h, w, 3] BGR on the device.  The engine must have been built with the depth
        map's own size as image size (the preview normalises the UN-resized map)."""
        if (self.dep_h, self.dep_w) != (self.img_h, self.img_w):
            raise ValueError("depth_preview needs an engine whose image size equals the depth size")
        from .plasma_lut import PLASMA_BGR
        if depth.device != self.device or depth.dtype != torch.float32 or not depth.is_contiguous() \
                or tuple(depth.shape) != (self.batch, self.dep_h, self.dep_w):
            raise ValueError("depth must be a contiguous float32 [batch, h, w] tensor on the engine's device")
        s = stream if stream is not None else torch.cuda.current_stream(self.device)
        cfg = self.make_config(density="high", invert=invert)
        with torch.cuda.device(self.device):
            if getattr(self, "_lut", None) is None:
                self._lut = torch.tensor(PLASMA_BGR, dtype=torch.uint8, device=self.device).contiguous()
            out = torch.empty((self.batch, self.dep_h, self.dep_w, 3), dtype=torch.uint8, device=self.device)

        def run():
            self._call("d2pc_preview_enqueue", C.byref(cfg), depth.data_ptr(), self.workspace.data_ptr(),
                       self.workspace_bytes, self._lut.data_ptr(), out.data_ptr(), s.cuda_stream)
        self.enqueue_stats(cfg, depth, s)
        self.enqueue_status(cfg, s)
        run()
        s.synchronize()
        if int(self._any_host[0]) != 0:
            self.enqueue_stats_fallback(cfg, depth, s)
            run()
            s.synchronize()
        return out

    # ---- whole path ----------------------------------------------------------------------
    def process(self, cfg: D2pcConfig, depth: torch.Tensor, bgr: Optional[torch.Tensor],
                xyz: Optional[torch.Tensor] = None, rgb: Optional[torch.Tensor] = None,
                count: Optional[torch.Tensor] = None, stream=None, smooth_ksize=None, after_emit=None) -> EmitResult:
        """stats -> emit for one device-resident batch; synchronises the stream once to learn
        whether any frame needs the exact fallback, and if so runs it and re-emits those frames.
        ``after_emit(xyz, rgb, count, bounds)`` is called after every emit has been enqueued and before the
        stream is synchronised (device -> host copies that should ride on the same synchronisation)."""
        self._check_inputs(depth, bgr)
        if xyz is None or rgb is None:
            xyz, rgb = self.alloc_outputs(cfg)
        n = self.points_per_frame(cfg)
        if tuple(xyz.shape) != (self.batch, n, 3) or tuple(rgb.shape) != (self.batch, n, 3):
            raise ValueError("output tensors must be float32 [batch, N, 3]")
        with torch.cuda.device(self.device):
            if count is None:
                count = torch.zeros(self.batch, dtype=torch.int32, device=self.device)
            bounds = torch.empty((self.batch, 6), dtype=torch.float32, device=self.device) if cfg.want_bounds else None
        s = stream if stream is not None else torch.cuda.current_stream(self.device)
        def emit():
            if smooth_ksize is None:
                self.enqueue_emit(cfg, depth, bgr, xyz, rgb, count, bounds, s)
            else:
                self.enqueue_emit_smooth(cfg, smooth_ksize, depth, bgr, xyz, rgb, count, bounds, s)
            if after_emit is not None:
                with torch.cuda.stream(s):
                    after_emit(xyz, rgb, count, bounds)
        if smooth_ksize is None:
            # statistics, status and emit in one library call
            self.enqueue_path(cfg, depth, bgr, xyz, rgb, count, bounds, s)
            if after_emit is not None:
                with torch.cuda.stream(s):
                    after_emit(xyz, rgb, count, bounds)
        else:
            self.enqueue_stats(cfg, depth, s)
            self.enqueue_status(cfg, s)
            emit()
        s.synchronize()
        if int(self._any_host[0]) != 0:
            # frames the fast statistics could not finish exactly: batch-wide statistics again (the pipeline
            # keeps only the last sub-batches' resized maps), the exact fallback for the flagged frames, emit
            self.enqueue_stats(cfg, depth, s)
            self.enqueue_stats_fallback(cfg, depth, s)
            emit()
            s.synchronize()
        return EmitResult(xyz, rgb, count, bounds)

    def frame_params(self, cfg: D2pcConfig):
        """Per-frame normalisation parameters as the device computed them (tests / debugging)."""
        with torch.cuda.device(self.device):
            buf = torch.zeros(self.batch * C.sizeof(D2pcFrameParams), dtype=torch.uint8, device=self.device)
        self._call("d2pc_frame_params", C.byref(cfg), self.workspace.data_ptr(), buf.data_ptr(), self._stream(None))
        raw = buf.cpu().numpy().tobytes()
        out = []
        for b in range(self.batch):
            p = D2pcFrameParams.from_buffer_copy(raw, b * C.sizeof(D2pcFrameParams))
            out.append({k: (list(getattr(p, k)) if k in ("n_cand", "reserved") else getattr(p, k))
                        for k, _ in D2pcFrameParams._fields_})
        return out

    # ---- ax-2 voxel grid ------------------------------------------------------------------
    def voxel_downsample(self, cfg: D2pcConfig, res: EmitResult, voxel_size: float,
                         want_index: bool = False, stream=None, check_error: bool = True):
        """Voxel-grid down-sampling of the emitted rows of every frame (needs cfg.want_bounds).
        Returns (vox_xyz [B,N,3], vox_rgb [B,N,3], vox_idx [B,N,3] or None, vox_count [B])."""
        if not cfg.want_bounds or res.bounds is None:
            raise ValueError("voxel_downsample needs an emit with want_bounds=True")
        if not voxel_size > 0:
            raise ValueError("voxel_size <= 0.")
        if not np.isfinite(voxel_size):
            raise ValueError("voxel_size must be finite.")
        nbytes = C.c_size_t(0)
        check(self.lib.d2pc_voxel_table_bytes(C.byref(cfg), C.byref(nbytes)), "d2pc_voxel_table_bytes")
        n = self.points_per_frame(cfg)
        with torch.cuda.device(self.device):
            if self._voxel_table is None or self._voxel_table.numel() < nbytes.value:
                self._voxel_table = torch.empty(int(nbytes.value), dtype=torch.uint8, device=self.device)
                self._voxel_rows = None
            if self._voxel_rows != n:   # the table's layout depends on the rows per frame (density)
                self._call("d2pc_voxel_table_init", C.byref(cfg), self._voxel_table.data_ptr(),
                           self._voxel_table.numel(), self._stream(stream))
                self._voxel_rows = n
            vxyz = torch.empty_like(res.xyz)
            vrgb = torch.empty_like(res.rgb)
            vidx = torch.empty(res.xyz.shape, dtype=torch.int32, device=self.device) if want_index else None
            vcount = torch.zeros(self.batch, dtype=torch.int32, device=self.device)
            verr = torch.zeros(self.batch, dtype=torch.int32, device=self.device)
        self._call("d2pc_voxel_enqueue", C.byref(cfg), float(voxel_size), res.xyz.data_ptr(), res.rgb.data_ptr(),
                   res.count.data_ptr(), res.bounds.data_ptr(), self._voxel_table.data_ptr(),
                   self._voxel_table.numel(), vxyz.data_ptr(), vrgb.data_ptr(), _ptr(vidx), vcount.data_ptr(),
                   verr.data_ptr(), self._stream(stream))
        if check_error:
            e = verr.cpu()
            if bool((e == 2).any()):
                raise RuntimeError("voxel table was not initialised")
            if bool((e != 0).any()):
                raise ValueError("voxel_size is too small.")
        return vxyz, vrgb, vidx, vcount


class BatchStream:
    """Steady-state processing of a sequence of device-resident batches on one GPU.

    The statistics of batch k+1 (sample / scan / select: two of them are short single-wave kernels)
    are enqueued on a high-priority stream while the emit of batch k (the long HBM-bound kernel)
    runs on another, so the latency-bound launches hide behind the bandwidth-bound one.  Two
    FrameEngines (two workspaces) alternate.  The "any frame needs the exact fallback" flags are
    collected per batch and must be checked by the caller after ``finish()`` (``needs_fallback``);
    flagged batches are re-run with ``FrameEngine.process``.
    """

    def __init__(self, img_h: int, img_w: int, dep_h=None, dep_w=None, *, batch: int, img_c: int = 3,
                 device=None, **knobs):
        self.engines = [FrameEngine(img_h, img_w, dep_h, dep_w, batch=batch, img_c=img_c, device=device)
                        for _ in range(2)]
        self.device = self.engines[0].device
        self.cfg = self.engines[0].make_config(**knobs)
        with torch.cuda.device(self.device):
            lo, hi = torch.cuda.Stream.priority_range()
            self.s_stats = torch.cuda.Stream(self.device, priority=hi)
            self.s_emit = torch.cuda.Stream(self.device, priority=lo)
            self.stats_done = [torch.cuda.Event() for _ in range(2)]
            self.emit_done = [torch.cuda.Event() for _ in range(2)]
        self.k = 0
        self.flags = []

    def submit(self, depth, bgr, xyz, rgb, count) -> None:
        """Enqueue one batch (all arguments are device tensors of the engine's shapes)."""
        i = self.k % 2
        eng = self.engines[i]
        if self.k >= 2:
            self.s_stats.wait_event(self.emit_done[i])  # the workspace is free once emit(k-2) is done
        eng.enqueue_stats(self.cfg, depth, self.s_stats)
        eng._call("d2pc_frame_status", C.byref(self.cfg), eng.workspace.data_ptr(), eng._status.data_ptr(),
                  eng._any.data_ptr(), self.s_stats.cuda_stream)
        with torch.cuda.device(self.device):
            flag = torch.zeros(1, dtype=torch.int32, pin_memory=True)
            with torch.cuda.stream(self.s_stats):
                flag.copy_(eng._any, non_blocking=True)
        self.flags.append(flag)
        self.stats_done[i].record(self.s_stats)
        self.s_emit.wait_event(self.stats_done[i])
        eng.enqueue_emit(self.cfg, depth, bgr, xyz, rgb, count, None, self.s_emit)
        self.emit_done[i].record(self.s_emit)
        self.k += 1

    def finish(self) -> None:
        self.s_stats.synchronize()
        self.s_emit.synchronize()

    def needs_fallback(self):
        """Indices of submitted batches in which at least one frame was flagged (after finish())."""
        return [j for j, f in enumerate(self.flags) if int(f[0]) != 0]


def shard_frames(n_frames: int, world_size: int, rank: int) -> range:
    """Contiguous block partition of frame indices over ranks (one rank per GPU, no collective:
    frames are independent).  Blocks differ by at most one frame."""
    if not (0 <= rank < world_size):
        raise ValueError("rank out of range")
    base, extra = divmod(n_frames, world_size)
    start = rank * base + min(rank, extra)
    return range(start, start + base + (1 if rank < extra else 0))
