"""TEST INFRASTRUCTURE ONLY -- CPU oracle for the depth-map -> coloured point-cloud stage.

This file is a NumPy *restatement* of the reference's hot path
(``/root/reference/backend/app.py:174-250``, ``depth_to_point_cloud``) and of the third-party
arithmetic that path calls into.  It is the checker the CUDA path is compared against; it is NOT
part of the product.  Only ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` /
``--impl reference`` legs of ``bench.py`` may import it.  The product package
(``image_to_pointcloud_b200``) never imports anything from ``oracle/``.

Parity pin
----------
The reference has no tests or golden vectors of its own (SURVEY.md section 4), and its results
depend on the versions of NumPy and OpenCV that happen to be installed
(``backend/requirements.txt`` pins nothing).  The oracle is therefore pinned to the reference
function *executed unmodified in the build container* (NumPy 2.3.5, OpenCV 4.13.0 with IPP):
``oracle/make_golden.py`` stores outputs of the reference itself under ``tests/golden/`` on every
branch, and ``tests/test_oracle_golden.py`` checks bit-equality of this restatement against them.

Third-party arithmetic restated here (none of it is vendored under /root/reference):

* ``cv2.resize(..., INTER_LINEAR)`` on float32 (``app.py:188``): OpenCV 4.13.0 wheels dispatch
  this to Intel IPP.  IPP is closed source; its arithmetic was recovered bit-exactly by
  experiment (see ``resize_bilinear``) and is checked against ``cv2.resize`` in the tests.
* ``np.percentile(d, [2, 98])`` (``app.py:197``): NumPy 2.3.5 ``_quantile``/``_lerp``
  (``numpy/lib/_function_base_impl.py``), method "linear".
* ``np.nanmedian`` (``app.py:195``), ``np.clip`` (``app.py:201``) and NEP-50 type promotion,
  which makes the normalised map float64 in the percentile branch.

The two north-star extensions that have no reference code (depth-range mask, voxel-grid
down-sampling) are specified here (``range_mask``, ``voxel_downsample``); for those the header
says what DESIGN.md says: **parity unpinned** (no reference implementation exists), the spec is
frozen by this file.
"""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np

F32 = np.float32
F64 = np.float64

DENSITY_STEP = {"low": 4, "medium": 2, "high": 1}  # app.py:226


# --------------------------------------------------------------------------------------------
# exact float32 fused multiply-add (NumPy has none)
# --------------------------------------------------------------------------------------------
def fmaf(a, b, c):
    """Correctly rounded float32 ``a*b + c`` (one rounding), element-wise.

    a*b is exact in float64 (24+24 significant bits).  The float64 sum s = fl(p + c) may be
    rounded; double rounding to float32 can only go wrong when s lands exactly on a float32
    tie, in which case the sign of the exact float64 rounding error (TwoSum) decides.
    """
    a = np.asarray(a, dtype=F32).astype(F64)
    b = np.asarray(b, dtype=F32).astype(F64)
    c = np.asarray(c, dtype=F32).astype(F64)
    with np.errstate(invalid="ignore", over="ignore"):
        p = a * b
        s = p + c
        bb = s - p
        err = (p - (s - bb)) + (c - bb)  # exact error of the float64 addition
        r = s.astype(F32)
        fin = np.isfinite(s) & np.isfinite(err) & (err != 0.0)
        if np.any(fin):
            rd = r.astype(F64)
            # neighbour of r on the other side of s
            other = np.nextafter(r, np.where(s > rd, F32(np.inf), F32(-np.inf)).astype(F32))
            mid = 0.5 * (rd + other.astype(F64))
            tie = fin & (s == mid) & (s != rd)
            toward_other = np.sign(err) == np.sign(other.astype(F64) - rd)
            r = np.where(tie & toward_other, other, r)
    return r.astype(F32)


# --------------------------------------------------------------------------------------------
# a1  resize to the image size (app.py:186-188) -- cv2.resize INTER_LINEAR, IPP float32 path
# --------------------------------------------------------------------------------------------
def _axis_taps(n_src: int, n_dst: int):
    """Source taps for one axis: (i0, i1, t32, clamped).  Coordinates in float64, weight cast to
    f32.  ``clamped`` marks destination indices whose source coordinate fell outside
    [0, n_src-1): there the output is a plain copy of tap 0 (no arithmetic, so a non-finite
    neighbour cannot leak in -- probed with inf/NaN inputs)."""
    scale = F64(n_src) / F64(n_dst)
    d = np.arange(n_dst, dtype=F64)
    f = (d + 0.5) * scale - 0.5
    i0 = np.floor(f)
    t = f - i0
    i0 = i0.astype(np.int64)
    low = i0 < 0
    i0 = np.where(low, 0, i0)
    t = np.where(low, 0.0, t)
    high = i0 >= n_src - 1
    i0 = np.where(high, n_src - 1, i0)
    t = np.where(high, 0.0, t)
    clamped = low | high
    i1 = np.where(clamped, i0, i0 + 1)
    return i0, i1, t.astype(F32), clamped


def resize_bilinear(depth: np.ndarray, out_h: int, out_w: int) -> np.ndarray:
    """Bit-exact model of ``cv2.resize(depth, (out_w, out_h), interpolation=cv2.INTER_LINEAR)``
    for float32 single-channel input as executed by the OpenCV 4.13.0 / IPP build
    (reference call site ``app.py:188``).

    Two taps per axis, no anti-aliasing.  Border positions (clamped coordinate) copy tap 0,
    except that in the four corner blocks (both coordinates clamped) a +-inf tap becomes NaN.
    Horizontal pass first,
    ``r = fmaf(S[x1] - S[x0], tx, S[x0])`` with the subtraction rounded to float32, then the
    vertical pass on those rows, ``out = fmaf(r1 - r0, ty, r0)``.
    """
    src = np.ascontiguousarray(depth, dtype=F32)
    h, w = src.shape
    if h == 1 or w == 1:
        return _resize_bilinear_generic(src, out_h, out_w)
    x0, x1, tx, cx = _axis_taps(w, out_w)
    y0, y1, ty, cy = _axis_taps(h, out_h)
    with np.errstate(invalid="ignore", over="ignore"):
        a = src[:, x0]
        b = src[:, x1]
        rows = np.where(cx[None, :], a, fmaf((b - a).astype(F32), tx[None, :], a))  # [h, out_w]
        r0 = rows[y0, :]
        r1 = rows[y1, :]
        out = np.where(cy[:, None], r0, fmaf((r1 - r0).astype(F32), ty[:, None], r0))
        # corner blocks (both coordinates clamped): IPP does run arithmetic there -- a +-inf
        # tap comes out as NaN (inf - inf); finite values are unchanged.
        corner = cy[:, None] & cx[None, :]
        out = np.where(corner & np.isinf(out), F32(np.nan), out)
    return np.ascontiguousarray(out, dtype=F32)


def _resize_bilinear_generic(src: np.ndarray, out_h: int, out_w: int) -> np.ndarray:
    """``cv2.resize(..., INTER_LINEAR)`` for a float32 source with a 1-pixel side (same call site,
    ``app.py:188``).  OpenCV 4.13.0 does not hand such sources to IPP; its own two-pass code runs
    (third-party: opencv/modules/imgproc/src/resize.cpp, ``resizeGeneric_`` with ``HResizeLinear`` /
    ``VResizeLinear``; not vendored in the reference, restated from the published source and pinned
    against cv2.resize of this container, tests/test_oracle_golden.py):

    * coordinates ``f = float32((d + 0.5) * scale - 0.5)``, ``s = floor(f)``, weight ``t = f - s`` in float32;
    * columns: ``s < 0 -> s = 0, t = 0``; from the first column with ``s + 1 >= w`` on, a plain copy of
      ``S[min(s, w - 1)]``; otherwise ``row = S[s] * (1 - t) + S[s + 1] * t`` (two products, one sum, each
      rounded to float32, no FMA);
    * rows: weights are NOT clamped, only the row indices are: ``out = R[clip(s)] * (1 - t) + R[clip(s + 1)] * t``
      (so a one-row source gives ``v * (1 - t) + v * t``, and ``inf * 0`` is NaN where ``t == 0``).
    """
    h, w = src.shape

    def coords(n_src, n_dst):
        scale = F64(n_src) / F64(n_dst)
        f = ((np.arange(n_dst, dtype=F64) + 0.5) * scale - 0.5).astype(F32)
        s = np.floor(f).astype(np.int64)
        t = (f - s.astype(F32)).astype(F32)
        return s, t

    sx, tx = coords(w, out_w)
    low = sx < 0
    sx = np.where(low, 0, sx)
    tx = np.where(low, F32(0), tx)
    copy = sx + 1 >= w                       # monotone in the column index: everything from xmax on
    x0 = np.minimum(sx, w - 1)
    x1 = np.minimum(sx + 1, w - 1)
    sy, ty = coords(h, out_h)
    y0 = np.clip(sy, 0, h - 1)
    y1 = np.clip(sy + 1, 0, h - 1)
    one = F32(1)
    with np.errstate(invalid="ignore", over="ignore"):
        a, b = src[:, x0], src[:, x1]
        blend = ((a * (one - tx)[None, :]).astype(F32) + (b * tx[None, :]).astype(F32)).astype(F32)
        rows = np.where(copy[None, :], a, blend)
        r0, r1 = rows[y0, :], rows[y1, :]
        out = ((r0 * (one - ty)[:, None]).astype(F32) + (r1 * ty[:, None]).astype(F32)).astype(F32)
    return np.ascontiguousarray(out, dtype=F32)


# --------------------------------------------------------------------------------------------
# a2  non-finite repair (app.py:191-196)
# --------------------------------------------------------------------------------------------
def nanmedian_f32(d: np.ndarray) -> np.float32:
    """``np.nanmedian`` of a float32 array: NaN dropped, +-inf kept; middle element, or
    ``f32(f32(a + b) / 2)`` of the two middle elements for an even count; NaN if nothing left."""
    flat = np.asarray(d, dtype=F32).ravel()
    flat = flat[~np.isnan(flat)]
    n = flat.size
    if n == 0:
        return F32(np.nan)
    s = np.sort(flat)
    if n % 2 == 1:
        return F32(s[n // 2])
    with np.errstate(invalid="ignore", over="ignore"):
        return F32(F32(s[n // 2 - 1] + s[n // 2]) / F32(2.0))


def repair_nonfinite(d: np.ndarray) -> np.ndarray:
    d = np.asarray(d, dtype=F32)
    finite = np.isfinite(d)
    if not finite.all():
        med = nanmedian_f32(d)
        d = np.where(finite, d, med).astype(F32)
    return d


# --------------------------------------------------------------------------------------------
# a3  percentiles (app.py:197) -- numpy 2.3.5 _quantile / _lerp, method "linear"
# --------------------------------------------------------------------------------------------
def percentile_ranks(n: int, q: float):
    """(lo, hi, gamma) of the 'linear' method: vi = (n-1)*q in float64."""
    vi = F64(n - 1) * F64(q)
    if vi >= n - 1:
        # _get_indexes sets both neighbours to -1 (the last element); gamma = vi - (-1)
        return n - 1, n - 1, F64(vi + 1.0)
    lo = int(np.floor(vi))
    return lo, lo + 1, F64(vi - F64(lo))


def lerp_f32_pair(a: np.float32, b: np.float32, g: np.float64) -> np.float64:
    """NumPy ``_lerp`` for float32 neighbours and a float64 weight."""
    with np.errstate(invalid="ignore", over="ignore"):
        diff = F32(F32(b) - F32(a))
        r = F64(a) + F64(diff) * g
        if g >= 0.5:
            r = F64(b) - F64(diff) * (F64(1.0) - g)
    return F64(r)


def percentiles_2_98(d: np.ndarray) -> Tuple[np.float64, np.float64]:
    """``np.percentile(d, [2, 98])`` restated: exact order statistics + float64 lerp.
    Any NaN in ``d`` makes both results NaN (NumPy sorts NaN last and poisons the slice)."""
    flat = np.asarray(d, dtype=F32).ravel()
    n = flat.size
    if np.isnan(flat).any():
        return F64(np.nan), F64(np.nan)
    s = np.sort(flat)
    out = []
    for q in (F64(2) / F64(100), F64(98) / F64(100)):
        lo, hi, g = percentile_ranks(n, q)
        out.append(lerp_f32_pair(s[lo], s[hi], g))
    return out[0], out[1]


# --------------------------------------------------------------------------------------------
# a2..a5  normalise (app.py:191-206)
# --------------------------------------------------------------------------------------------
def normalise_depth(depth_resized: np.ndarray, invert: bool):
    """Returns (d, info).  d is float64 in the percentile branch, float32 otherwise."""
    d = repair_nonfinite(depth_resized)
    p2, p98 = percentiles_2_98(d)
    branch = "pct"
    if p98 <= p2:
        p2, p98 = float(d.min()), float(d.max())
        branch = "minmax"
    if p98 > p2:
        if branch == "pct":
            # np.float64 scalars are strongly typed under NEP 50 -> float64 chain
            c = np.minimum(np.maximum(d.astype(F64), p2), p98)
            d = (c - p2) / (p98 - p2 + 1e-6)
        else:
            # Python floats are weak -> float32 chain; divisor rounded to float32 once
            lo, hi = F32(p2), F32(p98)
            c = np.minimum(np.maximum(d, lo), hi)
            d = ((c - lo).astype(F32) / F32(p98 - p2 + 1e-6)).astype(F32)
    else:
        branch = "zeros"
        d = np.zeros_like(d)
    if invert:
        d = 1.0 - d  # dtype preserved (python float is weak)
    return d, {"branch": branch, "p2": p2, "p98": p98}


# --------------------------------------------------------------------------------------------
# a6  optional smoothing (app.py:208-214) -- cv2.GaussianBlur(d, (k, k), 0), BORDER_REFLECT_101
# --------------------------------------------------------------------------------------------
_SMALL_GAUSSIAN = {
    1: [1.0],
    3: [0.25, 0.5, 0.25],
    5: [0.0625, 0.25, 0.375, 0.25, 0.0625],
    7: [0.03125, 0.109375, 0.21875, 0.28125, 0.21875, 0.109375, 0.03125],
    9: [4 / 256, 13 / 256, 30 / 256, 51 / 256, 60 / 256, 51 / 256, 30 / 256, 13 / 256, 4 / 256],
}


def smooth_kernel_size(smooth_ksize) -> int:
    """k = max(3, int(smooth_ksize) // 2 * 2 + 1)   (app.py:210)"""
    return max(3, int(smooth_ksize) // 2 * 2 + 1)


def gaussian_kernel(k: int) -> np.ndarray:
    """cv2.getGaussianKernel(k, 0, CV_64F) [external, OpenCV 4.x getGaussianKernelBitExact]: fixed
    tables for odd k <= 9 when sigma <= 0 (bit-exact here).  Larger k: sigma = k*0.15 + 0.35,
    t_i = exp(-0.125 * x_i^2 / sigma^2) with x_i = 2i - (k-1), normalised by 1 / (2*sum + 1).
    OpenCV evaluates that with its own soft-float exp; libm's exp can differ in the last bit, so for
    k >= 11 the coefficients (and the blur) are only accurate to ~1e-16 relative, not bit-pinned."""
    import math
    if k in _SMALL_GAUSSIAN:
        return np.array(_SMALL_GAUSSIAN[k], dtype=F64)
    sigma = k * 0.15 + 0.35
    scale2x = -0.125 / (sigma * sigma)
    n2 = (k - 1) // 2
    vals = [math.exp(float((2 * i - (k - 1)) ** 2) * scale2x) for i in range(n2)]
    total = 0.0
    for v in vals:
        total += v
    total = total * 2.0 + 1.0
    mul1 = 1.0 / total
    half = [v * mul1 for v in vals]
    return np.array(half + [mul1] + half[::-1], dtype=F64)


def _reflect101_taps(x: np.ndarray, r: int, axis: int):
    pad = [(r, r) if a == axis else (0, 0) for a in range(2)]
    xp = np.pad(x, pad, mode="reflect") if min(x.shape[axis], 2) > 1 or r == 0 else np.pad(x, pad, mode="edge")
    n = x.shape[axis]

    def tap(o):
        idx = [slice(None)] * 2
        idx[axis] = slice(r + o, r + o + n)
        return xp[tuple(idx)]
    return tap


def _fma64(a, b, c):
    """Correctly rounded float64 a*b + c via error-free transformations (TwoProduct by Dekker
    splitting, TwoSum), good for the magnitudes met here (no overflow / subnormals)."""
    a = np.asarray(a, F64); b = np.asarray(b, F64); c = np.asarray(c, F64)
    split = 134217729.0  # 2^27 + 1
    def two_prod(x, y):
        p = x * y
        xs = x * split; xh = xs - (xs - x); xl = x - xh
        ys = y * split; yh = ys - (ys - y); yl = y - yh
        e = ((xh * yh - p) + xh * yl + xl * yh) + xl * yl
        return p, e
    def two_sum(x, y):
        s = x + y
        bb = s - x
        e = (x - (s - bb)) + (y - bb)
        return s, e
    p, pe = two_prod(a, b)
    s, se = two_sum(p, c)
    # exact value = s + (pe + se); round-to-nearest of that: add the small terms, then fix ties
    t = pe + se
    r = s + t
    return r


def gaussian_blur_f64(d: np.ndarray, k: int) -> np.ndarray:
    """Bit-exact model of cv2.GaussianBlur(float64 HxW, (k,k), 0) as built in OpenCV 4.13.0 (AVX2
    dispatch), recovered by experiment: separable, rows first.
      row pass     x <  W - W%4 : s = k0*x0 ; s = fma(kj, xj, s) for j = 1..k-1   (vector body)
                   x >= W - W%4 : the same sum with separate multiply and add      (scalar tail)
      column pass  s = kc*x0 ; s = s + k(c+j) * (x(+j) + x(-j)) for j = 1..r       (no FMA)
    Border: BORDER_REFLECT_101."""
    d = np.ascontiguousarray(d, dtype=F64)
    kk = gaussian_kernel(k)
    r = k // 2
    H, W = d.shape
    tap = _reflect101_taps(d, r, 1)
    body = kk[0] * tap(-r)
    tail = kk[0] * tap(-r)
    for j in range(1, k):
        body = _fma64(kk[j], tap(j - r), body)
        tail = tail + kk[j] * tap(j - r)
    rows = body.copy()
    wb = W - W % 4
    rows[:, wb:] = tail[:, wb:]
    tap = _reflect101_taps(rows, r, 0)
    out = kk[r] * tap(0)
    for j in range(1, r + 1):
        out = out + kk[r + j] * (tap(j) + tap(-j))
    return out


def gaussian_blur_f32_approx(d: np.ndarray, k: int) -> np.ndarray:
    """float32 maps (min/max and zeros branches) go through a different OpenCV/IPP code path whose
    rounding is not modelled: exact float64 convolution rounded once (within ~2e-7 relative of
    cv2; the tests use a tolerance for this branch)."""
    kk = gaussian_kernel(k)
    r = k // 2
    x = np.ascontiguousarray(d, dtype=F64)
    tap = _reflect101_taps(x, r, 1)
    rows = sum(kk[j] * tap(j - r) for j in range(k))
    tap = _reflect101_taps(rows, r, 0)
    return sum(kk[j] * tap(j - r) for j in range(k)).astype(F32)


# --------------------------------------------------------------------------------------------
# a7  intrinsics (app.py:216-223)
# --------------------------------------------------------------------------------------------
def intrinsics(img_w: int, img_h: int, fov: Optional[float] = None):
    cx, cy = img_w / 2.0, img_h / 2.0
    if fov and fov > 0:
        f = (img_w / 2.0) / np.tan(np.deg2rad(fov) / 2.0)
    else:
        f = max(img_w, img_h) * 1.2
    return float(cx), float(cy), float(f)


# --------------------------------------------------------------------------------------------
# a0..a11 the whole stage, vectorised (bit-identical to the reference's double loop)
# --------------------------------------------------------------------------------------------
def depth_to_point_cloud(image: np.ndarray, depth: np.ndarray,
                         density: str = "medium",
                         invert: bool = True,
                         depth_scale: float = 10.0,
                         smooth: bool = False,
                         smooth_ksize: int = 5,
                         fov: Optional[float] = None,
                         return_info: bool = False):
    """Vectorised restatement of ``backend/app.py:174-250``.  Same positional signature."""
    smooth_ksize_arg = smooth_ksize
    img_h, img_w = image.shape[:2]
    dep_h, dep_w = depth.shape[:2]
    if (dep_h, dep_w) != (img_h, img_w):
        depth = resize_bilinear(depth, img_h, img_w)
    d, info = normalise_depth(np.asarray(depth).astype(F32), invert)
    if smooth:
        k = smooth_kernel_size(smooth_ksize_arg)
        d = gaussian_blur_f64(d, k) if d.dtype == F64 else gaussian_blur_f32_approx(d, k)
        info["smooth_exact"] = bool(d.dtype == F64)
    cx, cy, f = intrinsics(img_w, img_h, fov)
    step = DENSITY_STEP[density]  # KeyError for anything else, like the reference
    vs = np.arange(0, img_h, step)
    us = np.arange(0, img_w, step)
    dd = d[::step, ::step].astype(F64)
    z = dd * float(depth_scale)
    zz = np.where(z != 0.0, z, 1e-6)
    x = ((us.astype(F64) - cx)[None, :] * zz) / f
    y = ((vs.astype(F64) - cy)[:, None] * zz) / f
    pts = np.stack([x, y, z], axis=-1).reshape(-1, 3).astype(F32)
    if image.ndim == 3 and image.shape[2] >= 3:
        cols = image[::step, ::step, 2::-1][..., :3] if image.shape[2] == 3 else \
            image[::step, ::step, :3][..., ::-1]
        cols = np.ascontiguousarray(cols).reshape(-1, 3).astype(F32)
    else:
        cols = np.full((pts.shape[0], 3), 128.0, dtype=F32)
    if return_info:
        info.update(cx=cx, cy=cy, f=f, step=step)
        return pts, cols, info
    return pts, cols


def depth_to_point_cloud_loop(image, depth, density="medium", invert=True, depth_scale=10.0,
                              smooth=False, smooth_ksize=5, fov=None):
    """Loop-faithful restatement: same per-pixel Python loop as ``app.py:228-246``, used as the
    timing stand-in for the reference on machines where /root/reference is absent (its cost
    profile -- two list appends per pixel, then np.array -- is the reference's)."""
    img_h, img_w = image.shape[:2]
    dep_h, dep_w = depth.shape[:2]
    if (dep_h, dep_w) != (img_h, img_w):
        depth = resize_bilinear(depth, img_h, img_w)
    d, _ = normalise_depth(np.asarray(depth).astype(F32), invert)
    if smooth:
        raise NotImplementedError
    cx, cy, f = intrinsics(img_w, img_h, fov)
    step = DENSITY_STEP[density]
    points, colors = [], []
    for v in range(0, img_h, step):
        for u in range(0, img_w, step):
            z = float(d[v, u]) * float(depth_scale)
            x = (u - cx) * (z if z != 0.0 else 1e-6) / f
            y = (v - cy) * (z if z != 0.0 else 1e-6) / f
            points.append([x, y, z])
            if image.ndim == 3 and image.shape[2] >= 3:
                b, g, r = image[v, u][:3]
                colors.append([int(r), int(g), int(b)])
            else:
                colors.append([128, 128, 128])
    return np.array(points, dtype=F32), np.array(colors, dtype=F32)


# --------------------------------------------------------------------------------------------
# f2  depth preview (app.py:124-153), up to the colour-mapped uint8 image
# --------------------------------------------------------------------------------------------
def depth_preview_bgr(depth: np.ndarray, invert: bool, lut_bgr: np.ndarray) -> np.ndarray:
    """create_depth_preview up to (and including) cv2.applyColorMap: the normalisation of
    app.py:127-147 on the UN-resized map, ``(d * 255.0).astype(np.uint8)`` (app.py:150) and the
    256-entry colour-map lookup (app.py:153; ``lut_bgr`` = COLORMAP_PLASMA as a [256,3] table)."""
    d, _ = normalise_depth(np.asarray(depth).astype(F32), invert)
    with np.errstate(invalid="ignore"):
        img = (d * 255.0).astype(np.uint8)
    return lut_bgr[img]


# --------------------------------------------------------------------------------------------
# ax-1  depth-range mask + ordered compaction  (north-star extension, parity unpinned)
# --------------------------------------------------------------------------------------------
def range_mask(points: np.ndarray, z_min: float, z_max: float) -> np.ndarray:
    """keep = (z32 >= f32(z_min)) & (z32 <= f32(z_max)) on the float32 z that a11 emits."""
    z = points[:, 2]
    return (z >= F32(z_min)) & (z <= F32(z_max))


def apply_range_mask(points, colors, z_min, z_max):
    keep = range_mask(points, z_min, z_max)
    return points[keep], colors[keep], keep


# --------------------------------------------------------------------------------------------
# ax-2  voxel-grid down-sampling (north-star extension, parity unpinned)
# --------------------------------------------------------------------------------------------
VOXEL_INDEX_BITS = 21


def voxel_indices(points: np.ndarray, voxel_size: float) -> np.ndarray:
    """Open3D ``PointCloud::VoxelDownSample`` indexing [external, from the published source]:
    on float64 copies of the float32 points, vmin = min_xyz - 0.5*vs,
    idx = floor((p - vmin) / vs) per axis."""
    p = np.asarray(points, dtype=F32).astype(F64)
    vs = F64(voxel_size)
    vmin = p.min(axis=0) - vs * 0.5
    idx = np.floor((p - vmin[None, :]) / vs).astype(np.int64)
    if idx.size and idx.max() >= (1 << VOXEL_INDEX_BITS):
        raise ValueError("voxel_size is too small.")
    return idx


def voxel_downsample(points: np.ndarray, colors: np.ndarray, voxel_size: float):
    """Mean of member points and colours per occupied voxel.  Returns
    (points f32 [V,3], colors f32 [V,3], idx int64 [V,3]) sorted by packed voxel key."""
    if voxel_size <= 0:
        raise ValueError("voxel_size <= 0.")
    if len(points) == 0:
        z = np.zeros((0, 3), F32)
        return z, z.copy(), np.zeros((0, 3), np.int64)
    idx = voxel_indices(points, voxel_size)
    key = (idx[:, 0] << (2 * VOXEL_INDEX_BITS)) | (idx[:, 1] << VOXEL_INDEX_BITS) | idx[:, 2]
    uniq, inv, cnt = np.unique(key, return_inverse=True, return_counts=True)
    V = uniq.size
    out_p = np.zeros((V, 3), F64)
    out_c = np.zeros((V, 3), F64)
    p64 = points.astype(F64)
    c64 = colors.astype(F64)
    for k in range(3):
        out_p[:, k] = np.bincount(inv, weights=p64[:, k], minlength=V)
        out_c[:, k] = np.bincount(inv, weights=c64[:, k], minlength=V)
    out_p /= cnt[:, None]
    out_c /= cnt[:, None]
    mask = (1 << VOXEL_INDEX_BITS) - 1
    uidx = np.stack([uniq >> (2 * VOXEL_INDEX_BITS), (uniq >> VOXEL_INDEX_BITS) & mask,
                     uniq & mask], axis=1)
    return out_p.astype(F32), out_c.astype(F32), uidx


# --------------------------------------------------------------------------------------------
# comparison helpers
# --------------------------------------------------------------------------------------------

# --------------------------------------------------------------------------------------------
# f3  writer byte layouts and preview rows (backend/app.py:310-389, 495-506)
# --------------------------------------------------------------------------------------------
def preview_rows(points: np.ndarray, colors: np.ndarray, max_preview: int = 20000):
    """app.py:495-503: the strided rows that become the preview JSON (before ``.astype(float).tolist()``)."""
    if len(points) > max_preview:
        stride = max(1, len(points) // max_preview)
        pprev = points[::stride]
        cprev = colors[::stride] if colors is not None and len(colors) else np.zeros_like(pprev)
    else:
        pprev = points
        cprev = colors if colors is not None and len(colors) else np.zeros_like(points)
    return pprev, cprev


def xyz_text(points: np.ndarray, colors: np.ndarray) -> bytes:
    """The bytes save_xyz writes (app.py:383-387): the same f-string over the same numpy scalars."""
    lines = []
    for i in range(len(points)):
        x, y, z = points[i]
        r, g, b = colors[i] if len(colors) > 0 else [128, 128, 128]
        lines.append(f"{x:.6f} {y:.6f} {z:.6f} {int(r)} {int(g)} {int(b)}\n")
    return "".join(lines).encode("ascii")


LAS_RECORD_DTYPE = np.dtype([("X", "<i4"), ("Y", "<i4"), ("Z", "<i4"), ("intensity", "<u2"), ("bit_fields", "u1"),
                             ("classification", "u1"), ("scan_angle_rank", "i1"), ("user_data", "u1"),
                             ("point_source_id", "<u2"), ("red", "<u2"), ("green", "<u2"), ("blue", "<u2")])


def las_records(points: np.ndarray, colors: np.ndarray, scale: float = 0.01):
    """save_las (app.py:343-377) up to the point records: LAS 1.2 point format 2 (26 bytes).
    PARITY UNPINNED: laspy is not installed in the build container; this restates laspy 2.x's
    ``ScaledArrayView`` assignment, ``np.round((value - offset) / scale)`` cast to int32, from its
    published source.  Returns (records, offsets[3])."""
    assert LAS_RECORD_DTYPE.itemsize == 26
    offset = [float(points[:, 0].min()), float(points[:, 1].min()), float(points[:, 2].min())]
    rec = np.zeros(len(points), dtype=LAS_RECORD_DTYPE)
    for k, name in enumerate("XYZ"):
        # laspy keeps scale / offset as float64 arrays (header.scales / header.offsets), so the float32
        # coordinates are promoted and the arithmetic is float64
        q = np.round((np.array(points[:, k]) - np.float64(offset[k])) / np.float64(scale))
        if q.max() > np.iinfo(np.int32).max or q.min() < np.iinfo(np.int32).min:
            raise OverflowError("scaled coordinate out of int32 range")
        rec[name] = q.astype(np.int32)
    c = np.clip(colors, 0, 255).astype(np.uint16)
    rec["red"], rec["green"], rec["blue"] = c[:, 0] * 256, c[:, 1] * 256, c[:, 2] * 256
    return rec, offset


PLY_RECORD_DTYPE = np.dtype([("x", "<f8"), ("y", "<f8"), ("z", "<f8"), ("red", "u1"), ("green", "u1"), ("blue", "u1")])


def ply_records(points: np.ndarray, colors: np.ndarray) -> np.ndarray:
    """save_ply (app.py:329-341): the vertex records of Open3D's binary little-endian PLY.
    PARITY UNPINNED: Open3D is not installed here; restated from its published writer
    (``double x,y,z; uchar red,green,blue``, colour = round(clamp(c, 0, 1) * 255) of the float64 copy of
    ``colors / 255.0``, which NumPy evaluates in float32)."""
    assert PLY_RECORD_DTYPE.itemsize == 27
    rec = np.zeros(len(points), dtype=PLY_RECORD_DTYPE)
    rec["x"], rec["y"], rec["z"] = points[:, 0], points[:, 1], points[:, 2]
    c = (colors / 255.0).astype(np.float64)
    c8 = np.floor(np.clip(c, 0.0, 1.0) * 255.0 + 0.5).astype(np.uint8)
    rec["red"], rec["green"], rec["blue"] = c8[:, 0], c8[:, 1], c8[:, 2]
    return rec


PLY_HEADER = ("ply\nformat binary_little_endian 1.0\ncomment Created by Open3D\nelement vertex {n}\n"
              "property double x\nproperty double y\nproperty double z\n"
              "property uchar red\nproperty uchar green\nproperty uchar blue\nend_header\n")



# --------------------------------------------------------------------------------------------
# f1  statistical outlier removal (refine_point_cloud, backend/app.py:252-269)
# --------------------------------------------------------------------------------------------
def statistical_outlier_removal(points: np.ndarray, nb_neighbors: int = 20, std_ratio: float = 2.0):
    """Open3D ``PointCloud::RemoveStatisticalOutliers`` as called at app.py:262 (points as float64).
    PARITY UNPINNED: Open3D is not installed in the build container; this restates its published source
    (geometry/PointCloud.cpp): exact k-NN *including the query point itself* (nanoflann, squared
    distances accumulated axis by axis in float64), mean of the square roots summed in ascending order,
    ``cloud_mean`` / ``sq_sum`` over the points with mean > 0 but divided by the number of points that
    found neighbours, Bessel-corrected standard deviation, keep ``0 < mean < cloud_mean + std_ratio * std``.
    The k-NN distances come from scipy's cKDTree (exact, float64).
    Returns (kept indices int64, avg_distances float64 [N], (cloud_mean, std_dev, threshold))."""
    from scipy.spatial import cKDTree
    p = np.ascontiguousarray(points, dtype=F64)
    n = len(p)
    if n == 0:
        return np.zeros(0, np.int64), np.zeros(0, F64), (0.0, 0.0, 0.0)
    k = min(int(nb_neighbors), n)
    dist, _ = cKDTree(p).query(p, k=k)
    dist = dist.reshape(n, k)
    avg = np.cumsum(dist, axis=1)[:, -1] / k          # std::accumulate: sequential, ascending order
    valid = n                                           # every point finds at least itself
    pos = avg > 0
    cloud_mean = float(np.cumsum(np.where(pos, avg, 0.0))[-1]) / valid
    sq = np.where(pos, (avg - cloud_mean) * (avg - cloud_mean), 0.0)
    std_dev = float(np.sqrt(np.cumsum(sq)[-1] / (valid - 1))) if valid > 1 else float("nan")
    thr = cloud_mean + std_ratio * std_dev
    keep = np.nonzero(pos & (avg < thr))[0].astype(np.int64)
    return keep, avg, (cloud_mean, std_dev, thr)


def bit_equal(a: np.ndarray, b: np.ndarray) -> bool:
    a = np.ascontiguousarray(a)
    b = np.ascontiguousarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    return bool(np.array_equal(a.view(np.uint8), b.view(np.uint8)))


def count_bit_mismatch(a: np.ndarray, b: np.ndarray) -> int:
    a = np.ascontiguousarray(a, dtype=F32).view(np.uint32)
    b = np.ascontiguousarray(b, dtype=F32).view(np.uint32)
    return int((a != b).sum())
