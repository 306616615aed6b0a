"""Host plumbing of the device stages: device selection, uploads, scratch, the rows' bounds pass, error words and the
copies back to the host.  ``_lib`` stays the bare ctypes binding; this module is its torch side."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import check

_NUMPY_DTYPE = {torch.float32: np.float32, torch.float64: np.float64, torch.int32: np.int32, torch.int64: np.int64}


def device_for(x, device=None) -> torch.device:
    """The device a call on ``x`` runs on: the tensor's own, else ``device``, else the current CUDA device."""
    if not torch.cuda.is_available():
        raise RuntimeError("image_to_pointcloud_b200 needs a CUDA device (no CPU fallback exists)")
    if isinstance(x, torch.Tensor):
        return x.device
    return torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")


def upload(x, dtype: torch.dtype, cols: int, dev) -> torch.Tensor:
    """A NumPy array (cast to ``dtype``) or a tensor (which must have ``dtype``) as a contiguous [-1, cols] tensor on
    ``dev``, 1-D for ``cols=0``."""
    if isinstance(x, torch.Tensor):
        t = x.to(dev)
    else:
        t = torch.from_numpy(np.ascontiguousarray(x, dtype=_NUMPY_DTYPE[dtype])).to(dev)
    if t.dtype != dtype:
        raise ValueError(f"expected {dtype}, got {t.dtype}")
    return (t.reshape(-1, cols) if cols else t.reshape(-1)).contiguous()


def device_rows(points, colors, device=None):
    """-> (xyz [n,3] f32 cuda, rgb [n,3] f32 cuda, count int32 [1] cuda, n)"""
    dev = device_for(points, device)
    if isinstance(points, torch.Tensor):
        xyz = points
    else:
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


def stream(dev) -> int:
    return torch.cuda.current_stream(dev).cuda_stream


def ptr(t):
    """Device pointer of ``t``, None for None or an empty tensor (the C ABI takes NULL for an absent array)."""
    return t.data_ptr() if t is not None and t.numel() > 0 else None


def scratch(fn, *dims, dev) -> torch.Tensor:
    """The scratch a ``d2pc_*_scratch_bytes`` binding ``fn`` asks for at ``dims``, allocated on ``dev``."""
    nb = C.c_size_t(0)
    check(fn(*dims, C.byref(nb)), fn.__name__)
    return torch.empty(int(nb.value), dtype=torch.uint8, device=dev)


def row_bounds(xyz: torch.Tensor, count: torch.Tensor, n: int, dev) -> torch.Tensor:
    """min x, y, z, max x, y, z of the first ``count`` of ``n`` rows: float32 [6] on the device."""
    keys = torch.empty(6, dtype=torch.int32, device=dev)
    bounds = torch.empty(6, dtype=torch.float32, device=dev)
    check(_lib.load_library().d2pc_rows_bounds_enqueue(xyz.data_ptr(), count.data_ptr(), n, keys.data_ptr(),
                                                       bounds.data_ptr(), stream(dev)), "d2pc_rows_bounds_enqueue")
    return bounds


def raise_errors(err: int, table, where: str) -> None:
    """A device error word -> exceptions: the bits of ``table`` ((bit, message), ...) are errors in the input and raise
    ValueError with their messages; any other bit is a device loop that ran out of its bound (RuntimeError)."""
    known = 0
    for bit, _ in table:
        known |= bit
    if err & ~known:
        raise RuntimeError(f"{where}: a device loop exhausted its bound (error word {err})")
    if err:
        raise ValueError("; ".join(msg for bit, msg in table if err & bit))


def to_host(x, return_device: bool):
    """``x`` (a tensor, None, or a tuple or ``TriangleMesh`` of them) as it is with ``return_device``, else with
    every tensor copied to a NumPy array."""
    if return_device or x is None:
        return x
    if isinstance(x, tuple):
        parts = [to_host(t, False) for t in x]
        return type(x)(*parts) if hasattr(x, "_fields") else tuple(parts)
    return x.cpu().numpy()


def pinned(t: torch.Tensor) -> np.ndarray:
    """Device tensor -> a fresh C-contiguous NumPy array in pinned host memory (torch's caching host allocator, so the
    copy runs at PCIe speed; the array owns its buffer)."""
    host = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    host.copy_(t)
    return host.numpy()
