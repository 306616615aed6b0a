"""CPU: the voxel-grid reference and checker (row ax-2) pinned without a GPU, and the host side of the voxel ABI.

* The oracle (oracle.d2pc_oracle.voxel_downsample) against an independent per-point restatement of the spec: a dict
  keyed by the index tuple of the float64 formula, means by math.fsum, colours exact.  Same generators as the GPU
  tests (tests/voxel_cases.py).
* The checker the GPU tests use (voxel_cases.check_frame) accepts the oracle and refuses outputs that are subtly
  wrong: a colour one ulp off, an index off by one, a mean off by a few quanta of the fixed point.
* A NumPy model of the kernel's fixed-point sums: anchored at the cloud's minimum it meets the bound at any voxel
  size; anchored at vmin = min - vs/2 it does not once the voxel is much larger than the cloud.
* Host-only ABI checks: row limit and voxel_size validation happen before any launch."""
import ctypes as C
import math

import numpy as np
import pytest

from oracle import d2pc_oracle as O
from tests import voxel_cases as V

F32, F64 = np.float32, np.float64


def restated(xyz, rgb, vs):
    """The spec, one point at a time: vmin = min - vs/2; idx = floor((p - vmin) / vs) in float64; the mean of the
    members (math.fsum, then float32) and of their colours (exact integer sums)."""
    pts = [tuple(float(v) for v in row) for row in xyz]
    vmin = [min(p[a] for p in pts) - vs * 0.5 for a in range(3)]
    cells = {}
    for p, c in zip(pts, rgb):
        key = tuple(int(math.floor((p[a] - vmin[a]) / vs)) for a in range(3))
        cells.setdefault(key, []).append((p, c))
    out = {}
    for key, members in cells.items():
        n = len(members)
        mean = [math.fsum(p[a] for p, _ in members) / n for a in range(3)]
        col = [sum(int(c[a]) for _, c in members) / n for a in range(3)]
        out[key] = (np.array(mean, F64), np.array(col, F64).astype(F32), n)
    return out


def _clouds():
    rng = np.random.default_rng(11)
    out = {}
    for vs in (0.25, 0.1, 0.005, 1 / 3):
        for axis in range(3):
            out[f"faces vs={vs:.4g} axis={axis}"] = (V.face_cloud(vs, axis, rng, base=-1.5, faces=40), vs)
    out["limit 2^21-1 all axes"] = (V.limit_cloud(1.0, (0, 1, 2), V.IDX_LIMIT - 1, rng, n_fill=200), 1.0)
    out["limit 2^21-1 axis 1, vs 0.005"] = (V.limit_cloud(0.005, (1,), V.IDX_LIMIT - 1, rng, n_fill=200), 0.005)
    out["runs"] = (V.runs_cloud([1, 2, 31, 32, 33, 63, 64, 100], 0.01, rng, lead=5), 0.01)
    out["abab"] = (V.abab_cloud(300, 0.01, rng), 0.01)
    out["scattered"] = (V.scattered_cloud(2000, 0.01, rng, every=97), 0.01)
    out["lattice"] = (V.lattice_cloud(9, 1.0), 0.5)
    for name, p in V.degenerate_clouds(rng).items():
        for vs in (0.05, 1e3, 1e9, 1e300):
            out[f"{name} vs={vs:g}"] = (p[:1500], vs)
    for i in range(6):
        p, kind = V.random_cloud(rng, int(rng.choice([1, 40, 700, 2000])))
        out[f"random {i} {kind}"] = (p[:2500], V.fuzz_voxel_size(rng, p))
    return out


CLOUDS = _clouds()


@pytest.mark.parametrize("name", list(CLOUDS))
def test_oracle_matches_the_per_point_restatement(name):
    xyz, vs = CLOUDS[name]
    rgb = V.colours(np.random.default_rng(len(xyz)), len(xyz))
    want = restated(xyz, rgb, vs)
    p, c, idx = O.voxel_downsample(xyz, rgb, vs)
    assert len(p) == len(want)
    keys = [tuple(int(v) for v in row) for row in idx]
    assert keys == sorted(want), "voxel indices (sorted by packed key) differ from the restatement"
    mean = np.array([want[k][0] for k in keys])
    assert np.array_equal(c, np.array([want[k][1] for k in keys])), "colour means are not exact"
    # the oracle rounds its float64 mean to float32: within one float32 ulp of the exact mean
    assert np.all(np.abs(p.astype(F64) - mean) <= np.spacing(np.abs(mean).astype(F32)).astype(F64))
    # the extended-precision means the GPU tests use agree with math.fsum to far inside the bar
    ks, cnt, lmean, csum = V.exact_means(xyz, rgb, vs)
    assert np.array_equal(cnt, [want[k][2] for k in keys])
    assert np.all(np.abs(lmean.astype(F64) - mean) <= 2.0 ** -50 * (np.abs(mean) + V.extent(xyz)))
    # and the oracle's own output passes the checker
    problems, ratio = V.check_frame(p, c, idx.astype(np.int32), xyz, rgb, vs, name)
    assert problems == [] and ratio <= 1.0


def test_index_limit_in_the_oracle():
    rng = np.random.default_rng(12)
    for vs in (1.0, 0.005, 1 / 3):
        for axes in ((0,), (2,), (0, 1, 2)):
            ok = V.limit_cloud(vs, axes, V.IDX_LIMIT - 1, rng, n_fill=50)
            c = V.colours(rng, len(ok))
            assert int(O.voxel_downsample(ok, c, vs)[2].max()) == V.IDX_LIMIT - 1
            bad = V.limit_cloud(vs, axes, V.IDX_LIMIT, rng, n_fill=50)
            with pytest.raises(ValueError):
                O.voxel_downsample(bad, V.colours(rng, len(bad)), vs)


def test_face_clouds_straddle_the_faces():
    """The face generator does what the device test relies on: neighbouring float32 values land in different
    voxels of the tested axis."""
    rng = np.random.default_rng(13)
    for vs in (0.25, 0.1, 0.005, 1 / 3):
        for axis in range(3):
            p = V.face_cloud(vs, axis, rng, base=2.5, faces=30)
            idx = V.grid_index(p, vs)[1:, axis]   # rows come in groups of 7 around one face
            groups = idx.reshape(-1, 7)
            assert np.all(groups.max(axis=1) - groups.min(axis=1) == 1), (vs, axis)


def test_checker_refuses_subtly_wrong_outputs():
    rng = np.random.default_rng(14)
    xyz = V.one_voxel_cloud(5000, rng, size=10.0)
    xyz = np.concatenate([xyz, V.runs_cloud([3, 40, 7], 0.5, rng, lead=2) + np.float32(20.0)])
    rgb = V.colours(rng, len(xyz))
    vs = 1.0
    p, c, idx = O.voxel_downsample(xyz, rgb, vs)
    idx = idx.astype(np.int32)
    assert V.check_frame(p, c, idx, xyz, rgb, vs)[0] == []
    # a colour one float32 ulp off
    c2 = c.copy()
    c2[3, 1] = np.nextafter(c2[3, 1], F32(np.inf))
    assert V.check_frame(p, c2, idx, xyz, rgb, vs)[0]
    # an index off by one
    i2 = idx.copy()
    i2[5, 2] += 1
    assert V.check_frame(p, c, i2, xyz, rgb, vs)[0]
    # a voxel missing
    assert V.check_frame(p[1:], c[1:], idx[1:], xyz, rgb, vs)[0]
    # a mean off by 2^-36 of the extent (the fixed point promises 2^-38): refused even though rtol=1e-5 would pass
    E = V.extent(xyz)
    p2 = p.astype(F64)
    k = int(np.argmax(np.abs(p2[:, 0])))
    p2[k, 0] += max(2.0 ** -36 * E, 3 * float(np.spacing(np.abs(p[k, 0]))))
    p2 = p2.astype(F32)
    assert np.allclose(p2, p, rtol=1e-5, atol=1e-6)
    assert V.check_frame(p2, c, idx, xyz, rgb, vs)[0]
    # the row order does not matter
    perm = rng.permutation(len(p))
    assert V.check_frame(p[perm], c[perm], idx[perm], xyz, rgb, vs)[0] == []


def fixed_point_means(xyz, rgb, vs, origin="min"):
    """NumPy model of the kernel's coordinate means (csrc/d2pc_voxel.cu): per-frame power-of-two scale from the
    extent, 64-bit integer sums of round((p - origin) * scale), mean = origin + sum / scale / n, then float32.
    origin="min" is the frame's minimum with E = max(max - min); origin="vmin" is min - vs/2 with the extent
    measured from there (the half voxel included)."""
    p = xyz.astype(F64)
    bmin, bmax = p.min(axis=0), p.max(axis=0)
    org = bmin if origin == "min" else bmin - vs * 0.5
    ext = float((bmax - org).max())
    ex = math.frexp(ext)[1] if 0.0 < ext < 1e300 else 0
    scale = math.ldexp(1.0, 38 - ex)
    q = np.rint((p - org) * scale).astype(np.int64)
    keys = V.pack_key(V.grid_index(xyz, vs))
    order = np.argsort(keys, kind="stable")
    ks = keys[order]
    starts = np.flatnonzero(np.r_[True, ks[1:] != ks[:-1]])
    cnt = np.diff(np.r_[starts, len(ks)])
    sums = np.add.reduceat(q[order], starts, axis=0)
    return (org + (sums.astype(F64) / scale) / cnt[:, None]).astype(F32)


@pytest.mark.parametrize("vs", [0.05, 1e3, 1e7, 1e9])
def test_fixed_point_anchored_at_the_cloud_meets_the_bound(vs):
    """The kernel's arithmetic, restated: anchored at the cloud's minimum and scaled to its extent, the means meet
    2^-38 * E + ulp_f32 at every voxel size; anchored at vmin they lose it once vs is ~1e6 times the cloud."""
    rng = np.random.default_rng(15)
    xyz = V.degenerate_clouds(rng)["three_points"]
    rgb = V.colours(rng, len(xyz))
    _, c, idx = O.voxel_downsample(xyz, rgb, vs)
    good = fixed_point_means(xyz, rgb, vs, "min")
    assert V.check_frame(good, c, idx.astype(np.int32), xyz, rgb, vs)[0] == []
    old = fixed_point_means(xyz, rgb, vs, "vmin")
    assert bool(V.check_frame(old, c, idx.astype(np.int32), xyz, rgb, vs)[0]) == (vs >= 1e7)


# ---- host side of the ABI ----------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    import image_to_pointcloud_b200 as m
    return m.load_library()


def _cfg(h, w, step=1):
    import image_to_pointcloud_b200 as m
    return m.D2pcConfig(batch=1, img_h=h, img_w=w, img_c=3, dep_h=h, dep_w=w, step=step, invert=1,
                        depth_scale=10.0, cx=w / 2, cy=h / 2, f=1.2 * max(h, w), want_bounds=1)


def test_voxel_row_limit(lib):
    n = C.c_size_t(0)
    assert lib.d2pc_voxel_table_bytes(C.byref(_cfg(4095, 4096)), C.byref(n)) == 0
    assert n.value >= 4095 * 4096 * (4 * 2 + 8 + 40 + 1)
    assert lib.d2pc_voxel_table_bytes(C.byref(_cfg(4096, 4096)), C.byref(n)) == 4   # D2PC_ERR_UNSUPPORTED
    assert lib.d2pc_voxel_table_bytes(C.byref(_cfg(4096, 4096, step=2)), C.byref(n)) == 0   # N counts rows, not pixels


@pytest.mark.parametrize("vs", [0.0, -1.0, float("nan"), float("inf"), float("-inf")])
def test_voxel_enqueue_refuses_a_bad_voxel_size_before_any_launch(lib, vs):
    """Every pointer is set (never dereferenced on the host) and the table is too small: a valid voxel size reaches
    the size check (D2PC_ERR_WORKSPACE_TOO_SMALL) and returns before any launch, a bad one is refused first."""
    cfg = _cfg(64, 64)
    fake = C.c_void_p(1 << 20)

    def enqueue(v):
        return lib.d2pc_voxel_enqueue(C.byref(cfg), v, fake, fake, fake, fake, fake, 0, fake, fake, fake, fake,
                                      fake, None)
    assert enqueue(0.05) == 2
    assert enqueue(vs) == 1   # D2PC_ERR_INVALID_ARGUMENT
