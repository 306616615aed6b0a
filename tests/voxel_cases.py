"""Synthetic clouds built against the voxel grid (row ax-2, csrc/d2pc_voxel.cu), the high-precision reference
means, and the comparison shared by tests/test_voxel_cpu.py, tests/test_voxel_gpu.py and profiles/fuzz_voxel.py.

Every generator returns float32 xyz [n, 3] (C-contiguous); colours come from ``colours`` and are the integral
0..255 floats emit writes.  The grid is Open3D's: vmin = min_xyz - vs/2, idx = floor((p - vmin) / vs) on float64
copies, so a generator that wants to place points on a voxel face computes the face the same way.

The bar of ``check_frame``:
  * voxel count equal, indices bit-exact (after sorting both sides by packed key);
  * colour means bit-exact: both sides divide exact integer sums by n with a correctly rounded quotient;
  * coordinate means within 2^-38 * E + ulp_f32(mean) of the exact mean, E = max over axes of (max - min) of the
    cloud (no half voxel): what the 64-bit fixed point scaled to E promises (include/d2pc.h)."""
from __future__ import annotations

import numpy as np

from oracle import d2pc_oracle as O

F32, F64 = np.float32, np.float64
BITS = O.VOXEL_INDEX_BITS
IDX_LIMIT = 1 << BITS


# --------------------------------------------------------------------------------------------
# helpers
# --------------------------------------------------------------------------------------------
def pack_key(idx: np.ndarray) -> np.ndarray:
    idx = np.asarray(idx, dtype=np.int64)
    return (idx[:, 0] << (2 * BITS)) | (idx[:, 1] << BITS) | idx[:, 2]


def grid_index(xyz: np.ndarray, vs: float) -> np.ndarray:
    """The oracle's float64 index formula, without its range check (generators aim at exact indices)."""
    p = np.asarray(xyz, dtype=F32).astype(F64)
    vmin = p.min(axis=0) - F64(vs) * 0.5
    return np.floor((p - vmin) / F64(vs)).astype(np.int64)


def bounds_of(xyz: np.ndarray) -> np.ndarray:
    """float32 [6]: min xyz then max xyz, the layout emit writes."""
    if len(xyz) == 0:
        return np.zeros(6, F32)
    return np.concatenate([xyz.min(axis=0), xyz.max(axis=0)]).astype(F32)


def extent(xyz: np.ndarray) -> float:
    """E = max over axes of (max - min): the cloud's own extent, without the half voxel."""
    if len(xyz) == 0:
        return 0.0
    b = bounds_of(xyz).astype(F64)
    return float((b[3:] - b[:3]).max())


def colours(rng, n: int, kind: str = "random") -> np.ndarray:
    if kind == "white":
        return np.full((n, 3), 255.0, F32)
    if kind == "black_white":
        return (rng.integers(0, 2, (n, 3)) * 255).astype(F32)
    return rng.integers(0, 256, (n, 3)).astype(F32)


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=F64).astype(F32))


def _ulps(x32: np.float32, k: int) -> np.float32:
    """The float32 k steps above (k > 0) or below (k < 0) x32."""
    d = F32(np.inf) if k > 0 else F32(-np.inf)
    for _ in range(abs(k)):
        x32 = np.nextafter(x32, d)
    return x32


# --------------------------------------------------------------------------------------------
# generators
# --------------------------------------------------------------------------------------------
def face_cloud(vs: float, axis: int, rng, base: float = 0.0, faces: int = 150, ulps: int = 3) -> np.ndarray:
    """Points at the float32 values nearest to the voxel faces vmin + k*vs of one axis, and their float32
    neighbours up to ``ulps`` steps on both sides: the floor of (p - vmin) / vs flips between them.  Row 0 is the
    anchor at ``base`` on every axis (the minimum, hence vmin = base - vs/2); the other axes stay inside a few
    voxels."""
    b0 = F32(base)
    vmin = F64(b0) - F64(vs) * 0.5
    ks = np.unique(np.r_[1, 2, 3, rng.integers(1, 4000, faces - 3)])
    vals = []
    for k in ks:
        c = F32(vmin + F64(k) * F64(vs))
        vals.extend(_ulps(c, j) for j in range(-ulps, ulps + 1))
    vals = np.array(vals, F32)
    vals = vals[vals > b0]
    p = np.empty((len(vals) + 1, 3), F32)
    p[0] = b0
    p[1:] = _f32(F64(b0) + rng.random((len(vals), 3)) * 3 * vs)
    p[1:, axis] = vals
    return np.ascontiguousarray(p)


def limit_cloud(vs: float, axes, imax: int, rng, n_fill: int = 500) -> np.ndarray:
    """A cloud whose largest index on each of ``axes`` is exactly ``imax``, reached by the largest float32 that
    still floors to ``imax`` (the voxel's upper face from below).  Row 0 is the anchor at 0."""
    idx_of = lambda v: int(np.floor((F64(v) + F64(vs) * 0.5) / F64(vs)))   # vmin = -vs/2
    p = F32(F64(imax) * F64(vs))
    while idx_of(p) > imax:
        p = _ulps(p, -1)
    while idx_of(p) < imax:
        p = _ulps(p, 1)
    while idx_of(_ulps(p, 1)) == imax:
        p = _ulps(p, 1)
    hi = F64(p)
    fill = _f32(rng.random((n_fill, 3)) * hi)
    out = np.concatenate([np.zeros((1, 3), F32), fill, np.zeros((2, 3), F32)])
    for a in axes:
        out[-2, a] = p
        out[-1, a] = _ulps(p, -1)
    assert int(grid_index(out, vs)[:, list(axes)].max()) == imax
    return np.ascontiguousarray(out)


def runs_cloud(lengths, vs: float, rng, lead: int = 5) -> np.ndarray:
    """Consecutive runs of rows in one voxel each, of the given lengths, after ``lead`` singleton rows so that the
    runs straddle 32-row groups and 1024-row tiles.  Row 0 is the anchor at 0 (voxel 0 spans (-vs/2, vs/2))."""
    rows = [np.zeros((1, 3))]
    cells = rng.permutation(200 ** 3)[: lead + len(lengths)]
    cells = np.stack([cells // 40000, (cells // 200) % 200, cells % 200], 1) + 1   # voxel (1..200)^3, never 0
    for j, c in enumerate(cells):
        n = 1 if j < lead else int(lengths[j - lead])
        rows.append((c + (rng.random((n, 3)) - 0.5) * 0.8) * vs)
    return _f32(np.concatenate(rows))


def abab_cloud(n: int, vs: float, rng) -> np.ndarray:
    """Two voxels alternating row by row: no run longer than 1, every row after the first two is a member."""
    c = np.array([[3, 4, 5], [3, 4, 6]])
    p = (c[np.arange(n) % 2] + (rng.random((n, 3)) - 0.5) * 0.8) * vs
    return _f32(np.concatenate([np.zeros((1, 3)), p]))


def scattered_cloud(n: int, vs: float, rng, every: int = 997) -> np.ndarray:
    """Every row its own voxel, except one voxel whose members sit every ``every`` rows (across many tiles)."""
    side = int(np.ceil((n + 1) ** (1 / 3))) + 1
    cell = np.stack(np.meshgrid(*[np.arange(1, side + 1)] * 3, indexing="ij"), -1).reshape(-1, 3)[:n]
    cell[::every] = (side + 3, side + 3, side + 3)
    p = (cell + (rng.random((n, 3)) - 0.5) * 0.8) * vs
    return _f32(np.concatenate([np.zeros((1, 3)), p]))


def one_voxel_cloud(n: int, rng, size: float = 10.0, offset=(0.0, 0.0, 0.0)) -> np.ndarray:
    """n random points in a box of side ``size``: one voxel for any vs > 2 * size."""
    return _f32(np.asarray(offset) + rng.random((n, 3)) * size)


def lattice_cloud(side: int, spacing: float = 1.0) -> np.ndarray:
    """side^3 points on a lattice in raster order; with vs = spacing / 2 every row is its own voxel."""
    g = np.arange(side, dtype=F64) * spacing
    return _f32(np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3))


def degenerate_clouds(rng) -> dict:
    """One point, three points near (0, 0, 3), identical points, a plane, a line, a cloud with every coordinate
    negative, tight clusters (about 10 units across where they have an extent)."""
    t = rng.random(400)
    return {
        "one_point": _f32([[1.25, -3.5, 7.0]]),
        "three_points": _f32([[0.1, -0.2, 3.0], [0.05, 0.3, 3.1], [-0.15, 0.01, 2.95]]),
        "identical": _f32(np.tile([[0.3, 0.2, 5.1]], (777, 1))),
        "plane": _f32(np.c_[rng.random((3000, 2)) * 10, np.full(3000, 2.5)]),
        "line": _f32(np.c_[t * 10, t * -4 + 1, np.full(400, -0.75)]),
        "negative": _f32(-(rng.random((5000, 3)) * 10 + 0.5)),
        "clusters": _f32((rng.random((40, 3)) * 10)[rng.integers(40, size=6000)] + rng.standard_normal((6000, 3)) * 0.01),
    }


def random_cloud(rng, n: int):
    """One cloud of a random kind (for the fuzz driver): (xyz, kind)."""
    kind = str(rng.choice(["uniform", "clusters", "plane", "line", "duplicates", "negative", "faces", "runs",
                           "lattice", "far"]))
    scale = float(rng.choice([1e-3, 0.1, 1.0, 10.0, 1e3]))
    if kind == "uniform":
        p = rng.random((n, 3)) * scale
    elif kind == "clusters":
        p = (rng.random((max(1, n // 100), 3)) * scale)[rng.integers(max(1, n // 100), size=n)]
        p = p + rng.standard_normal((n, 3)) * scale * 1e-3
    elif kind == "plane":
        p = np.c_[rng.random((n, 2)) * scale, np.full(n, float(rng.uniform(-5, 5)))]
    elif kind == "line":
        t = rng.random(n)
        p = np.c_[t * scale, t * -scale / 3, t * 0.0 + 1.0]
    elif kind == "duplicates":
        p = (rng.random((max(1, n // 7), 3)) * scale)[rng.integers(max(1, n // 7), size=n)]
    elif kind == "negative":
        p = -(rng.random((n, 3)) * scale + scale)
    elif kind == "far":   # a small cloud far from the origin: the fixed point must follow the cloud, not 0
        p = rng.random((n, 3)) * scale * 1e-3 + float(rng.choice([1e3, -4e4, 1e5]))
    elif kind == "faces":
        vs = float(rng.choice([0.25, 0.1, 0.005, 1 / 3]))
        p = face_cloud(vs, int(rng.integers(3)), rng, base=float(rng.uniform(-5, 5)), faces=max(4, n // 7))
    elif kind == "runs":
        lengths = rng.choice([1, 2, 31, 32, 33, 63, 64, 100, 1023, 1024, 1025], size=max(1, n // 300))
        p = runs_cloud(lengths, 0.01, rng, lead=int(rng.integers(0, 40)))
    else:
        p = lattice_cloud(max(1, int(round(n ** (1 / 3)))), scale)
    p = _f32(p)
    return (p if kind in ("faces", "runs") else p[:max(1, n)]), kind


def fuzz_voxel_size(rng, xyz) -> float:
    """A voxel size between ~1e-4 of the cloud's extent and far beyond it (never so small that indices overflow)."""
    e = max(extent(xyz), 1e-6)
    return float(e * 10.0 ** rng.uniform(-4.5, 1.0)) if rng.random() < 0.9 else float(rng.choice([0.25, 0.1, 0.005, 1 / 3]))


# --------------------------------------------------------------------------------------------
# reference and comparison
# --------------------------------------------------------------------------------------------
def exact_means(xyz: np.ndarray, rgb: np.ndarray, vs: float):
    """(keys int64 [V] ascending, counts [V], coordinate means longdouble [V, 3], colour sums int64 [V, 3]).
    Coordinate sums are taken in extended precision over key-sorted rows (np.add.reduceat): with n < 2^24 members
    their error is below 2^-40 of the summed magnitudes, far inside the bar."""
    keys = pack_key(grid_index(xyz, vs))
    order = np.argsort(keys, kind="stable")
    ks = keys[order]
    starts = np.flatnonzero(np.r_[True, ks[1:] != ks[:-1]])
    cnt = np.diff(np.r_[starts, len(ks)])
    p = xyz[order].astype(np.longdouble)
    mean = np.add.reduceat(p, starts, axis=0) / cnt[:, None].astype(np.longdouble)
    csum = np.add.reduceat(rgb[order].astype(np.int64), starts, axis=0)
    return ks[starts], cnt, mean, csum


def mean_bound(xyz: np.ndarray, mean: np.ndarray) -> np.ndarray:
    """2^-38 * E + ulp_f32(mean), per coordinate.  The first term is the fixed point's rounding (at most half a
    quantum per member, and the quantum is 2^(ex - 38) with E >= 2^(ex - 1)); the second covers the final
    rounding to float32.  The 2^-12 relative slack on the first term covers the two float64 roundings of the
    extract (sum -> double, quotient), each at most 2^-53 * E."""
    E = extent(xyz)
    ulp = np.spacing(np.abs(mean.astype(F64)).astype(F32)).astype(F64)
    return (2.0 ** -38) * E * (1 + 2.0 ** -12) + ulp


def check_frame(got_xyz, got_rgb, got_idx, xyz, rgb, vs: float, what: str = ""):
    """Problems of one frame's device output against the oracle and the exact means ([] = all held).
    Returns (problems, worst |error| / bound)."""
    problems = []
    want_p, want_c, want_idx = O.voxel_downsample(xyz, rgb, vs)
    if len(got_xyz) != len(want_p):
        return [f"{what}: {len(got_xyz)} voxels, oracle {len(want_p)}"], float("inf")
    if len(want_p) == 0:
        return [], 0.0
    gk = pack_key(got_idx)
    order = np.argsort(gk, kind="stable")
    if not np.array_equal(gk[order], pack_key(want_idx)):
        return [f"{what}: voxel indices differ from the oracle"], float("inf")
    gp, gc = got_xyz[order], got_rgb[order]
    if not np.array_equal(gc.view(np.uint32), want_c.view(np.uint32)):
        problems.append(f"{what}: colour means not bit-exact ({int((gc != want_c).sum())} words)")
    keys, cnt, mean, csum = exact_means(xyz, rgb, vs)
    assert np.array_equal(keys, pack_key(want_idx))
    # the oracle's colours are the correctly rounded quotients of the exact integer sums
    assert np.array_equal((csum / cnt[:, None]).astype(F32), want_c)
    err = np.abs(gp.astype(np.longdouble) - mean).astype(F64)
    bound = mean_bound(xyz, mean)
    ratio = float((err / bound).max())
    if ratio > 1.0:
        i = np.unravel_index(int(np.argmax(err / bound)), err.shape)
        problems.append(f"{what}: mean off by {err[i]:.3e} > bound {bound[i]:.3e} (voxel {i[0]} of {len(cnt)}, "
                        f"axis {i[1]}, {int(cnt[i[0]])} members, E = {extent(xyz):.6g}, vs = {vs:.6g})")
    return problems, ratio


def canonical(got_xyz, got_rgb, got_idx) -> bytes:
    """Bytes of one frame's output in packed-key order (for run-to-run / fused-vs-split comparisons)."""
    order = np.argsort(pack_key(got_idx), kind="stable")
    return got_xyz[order].tobytes() + got_rgb[order].tobytes() + np.asarray(got_idx)[order].tobytes()


# --------------------------------------------------------------------------------------------
# device harness (needs torch and a GPU; imported lazily so the CPU tests need neither)
# --------------------------------------------------------------------------------------------
def run_device(eng, cfg, frames, vs: float, split: bool = False):
    """Feed per-frame clouds [(xyz, rgb), ...] (at most eng.batch; missing frames are empty) straight into
    FrameEngine.voxel_downsample.  Rows past each frame's count are NaN / -1: they must never be read.
    Returns [(xyz, rgb, idx), ...] per frame and the raw vcount.  ``split`` selects the two-launch insert."""
    import os

    import torch

    from image_to_pointcloud_b200.engine import EmitResult
    B, N = eng.batch, eng.points_per_frame(cfg)
    xyz = np.full((B, N, 3), np.nan, F32)
    rgb = np.full((B, N, 3), -1.0, F32)
    cnt = np.zeros(B, np.int32)
    bnd = np.zeros((B, 6), F32)
    for b, (p, c) in enumerate(frames):
        assert len(p) <= N, (len(p), N)
        xyz[b, :len(p)] = p
        rgb[b, :len(p)] = c
        cnt[b] = len(p)
        bnd[b] = bounds_of(p)
    dev = eng.device
    res = EmitResult(torch.from_numpy(xyz).to(dev), torch.from_numpy(rgb).to(dev), torch.from_numpy(cnt).to(dev),
                     torch.from_numpy(bnd).to(dev))
    del xyz, rgb
    old = os.environ.get("D2PC_VOX_SPLIT")
    os.environ["D2PC_VOX_SPLIT"] = "1" if split else "0"
    try:
        vx, vr, vi, vc = eng.voxel_downsample(cfg, res, vs, want_index=True)
        torch.cuda.synchronize(dev)
    finally:
        if old is None:
            del os.environ["D2PC_VOX_SPLIT"]
        else:
            os.environ["D2PC_VOX_SPLIT"] = old
    vc = vc.cpu().numpy()
    out = []
    for b in range(B):
        n = int(vc[b])
        out.append((vx[b, :n].cpu().numpy(), vr[b, :n].cpu().numpy(), vi[b, :n].cpu().numpy()))
    return out, vc
