"""GPU (-m gpu): point normals (estimate_normals, Open3D semantics) against the oracle's restatement
(oracle/d2pc_normals_oracle.py).  Covariances are bit-exact (float64 words); normals agree to 1e-9 rad wherever the
two smallest eigenvalues are separated (acos / cos of libdevice and libm differ in the last ulps), are unit length
or exactly (0, 0, +-1), face the camera, and repeat bit for bit."""
import warnings

import numpy as np
import pytest

from oracle import d2pc_normals_oracle as N
from oracle import d2pc_oracle as O
from tests import cases

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def m():
    import torch
    assert torch.cuda.is_available()
    import image_to_pointcloud_b200 as mod
    mod.load_library()
    return mod


def _upper(cov33):
    return np.ascontiguousarray(np.asarray(cov33)[:, [0, 0, 0, 1, 1, 2], [0, 1, 2, 1, 2, 2]])


def _check(m, p, knn=30, radius=None, cam=(0.0, 0.0, 0.0)):
    """device vs oracle on one cloud; returns the device normals"""
    want_n, want_c = N.estimate_normals(p, knn=knn, radius=radius, orient_towards=cam, return_covariances=True)
    got_n, got_c = m.estimate_normals(p, knn=knn, radius=radius, orient_towards=cam, return_covariances=True)
    what = f"n={len(p)} knn={knn} radius={radius}"
    assert got_n.dtype == np.float64 and got_n.shape == (len(p), 3) and got_c.shape == (len(p), 3, 3), what
    gc = _upper(got_c)
    assert (gc.view(np.uint64) == want_c.view(np.uint64)).all(), \
        f"{what}: {(gc.view(np.uint64) != want_c.view(np.uint64)).any(1).sum()} covariances differ"
    # degenerate rows (identity covariance, zero covariance, axis-aligned) give an axis exactly; the rest unit length
    axis = (np.abs(got_n) == 1.0).sum(1) == 1
    assert np.allclose(np.linalg.norm(got_n[~axis], axis=1), 1.0, rtol=0, atol=1e-15), what
    ident = (want_c == [1, 0, 0, 1, 0, 1]).all(1) | (want_c == 0).all(1)
    assert (np.abs(got_n[ident]) == [0, 0, 1]).all(), what
    # angle to the oracle's normal where the smallest eigenvalue is separated
    w = np.linalg.eigvalsh(got_c)
    with np.errstate(all="ignore"):
        relgap = (w[:, 1] - w[:, 0]) / w[:, 2]
    sep = relgap >= 1e-6
    ang = np.arctan2(np.linalg.norm(np.cross(got_n, want_n), axis=1), np.abs((got_n * want_n).sum(1)))
    assert ang[sep].max(initial=0.0) <= 1e-9, f"{what}: max angle {ang[sep].max()}"
    # orientation: every row faces the camera; the sign agrees with the oracle away from n . (c - p) == 0
    if cam is not None:
        ref = np.asarray(cam, np.float64) - p.astype(np.float64)
        dot = (got_n * ref).sum(1)
        assert (dot >= 0).all(), what
        clear = sep & (np.abs(dot) > 1e-6 * np.linalg.norm(ref, axis=1))
        assert ((got_n * want_n).sum(1)[clear] > 0).all(), what
    # run to run
    again = m.estimate_normals(p, knn=knn, radius=radius, orient_towards=cam)
    assert again.tobytes() == got_n.tobytes(), what
    return got_n


def _stage_cloud(H, W, kind, density, seed=11):
    rng = np.random.default_rng(seed)
    img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return O.depth_to_point_cloud(img, cases.make_depth(H, W, seed, kind), density=density, invert=False)


@pytest.mark.parametrize("kind", ["uniform", "scene", "ties"])
@pytest.mark.parametrize("density", ["high", "medium"])
def test_normals_on_stage_outputs(m, kind, density):
    p, _ = _stage_cloud(120, 160, kind, density)
    _check(m, p)


def test_normals_on_a_larger_stage_cloud_with_heavy_cells(m):
    # 240 x 320 at density high: the clipped pixels form one cell of several thousand points (x-sorted walk)
    p, _ = _stage_cloud(240, 320, "scene", "high")
    _check(m, p)
    _check(m, p, knn=64)


@pytest.mark.parametrize("knn", [1, 3, 20, 30, 64])
def test_normals_knn_values(m, knn):
    rng = np.random.default_rng(20 + knn)
    blob = rng.standard_normal((4000, 3)).astype(np.float32)
    blob[:40] *= 30
    _check(m, blob, knn=knn)
    p, _ = _stage_cloud(96, 128, "ties", "high", seed=3)
    _check(m, p, knn=knn)


def test_normals_synthetic_clouds(m):
    rng = np.random.default_rng(30)
    blob = rng.standard_normal((5000, 3)).astype(np.float32)
    blob[:50] *= 30
    _check(m, blob)
    plane = np.c_[rng.random((3000, 2)) * 4, np.full(3000, 2.0)].astype(np.float32)
    assert np.allclose(_check(m, plane), [0, 0, -1], atol=1e-12)
    t = rng.random(800)
    line = (t[:, None] * [7.0, -3.0, 0.5] + [1.0, 2.0, 3.0]).astype(np.float32)
    _check(m, line, knn=10)
    dup = np.repeat(rng.standard_normal((60, 3)).astype(np.float32), 25, axis=0)
    _check(m, dup)
    lattice = (np.stack(np.meshgrid(*[np.arange(12)] * 3, indexing="ij"), -1).reshape(-1, 3) * 0.25).astype(np.float32)
    _check(m, lattice)
    _check(m, lattice, knn=7, cam=None)
    for n in (1, 2, 3, 29, 30, 31):
        _check(m, rng.standard_normal((n, 3)).astype(np.float32))
    _check(m, blob[:2000], cam=(3.0, -1.0, 40.0))


def test_normals_radius_mode(m):
    rng = np.random.default_rng(40)
    blob = rng.standard_normal((4000, 3)).astype(np.float32)
    blob[:40] *= 30
    lattice = (np.stack(np.meshgrid(*[np.arange(10)] * 3, indexing="ij"), -1).reshape(-1, 3) * 0.25).astype(np.float32)
    for radius, knn in ((0.05, 30), (0.2, 30), (0.5, 64), (5.0, 20)):
        _check(m, blob, knn=knn, radius=radius)     # small radii leave many points with < 3 neighbours
    for radius in (0.25, 0.2500001, 0.4, 0.6):       # exactly the spacing (strict d2 < r^2), just above, diagonals
        _check(m, lattice, knn=30, radius=radius)
    p, _ = _stage_cloud(120, 160, "scene", "high")
    _check(m, p, knn=30, radius=0.05)


def test_device_tensors_in_and_out(m):
    import torch
    rng = np.random.default_rng(50)
    p = rng.standard_normal((3000, 3)).astype(np.float32)
    t = torch.from_numpy(p).cuda()
    n, c = m.estimate_normals(t, return_covariances=True, return_device=True)
    assert n.is_cuda and c.is_cuda and n.dtype == torch.float64 and tuple(c.shape) == (3000, 3, 3)
    hn, hc = m.estimate_normals(p, return_covariances=True)
    assert n.cpu().numpy().tobytes() == hn.tobytes() and c.cpu().numpy().tobytes() == hc.tobytes()
    assert m.estimate_normals(np.zeros((0, 3), np.float32)).shape == (0, 3)
    bad = p.copy()
    bad[7, 2] = np.nan
    with pytest.raises(ValueError):
        m.estimate_normals(bad)
    with pytest.raises(ValueError):
        m.estimate_normals(p, knn=65)
    with pytest.raises(ValueError):
        m.estimate_normals(p, radius=-1.0)


def test_ply_with_normals_bytes(m, tmp_path, monkeypatch):
    p, c = cases.writer_rows(8, 5000)
    rng = np.random.default_rng(60)
    nrm = rng.standard_normal((5000, 3))
    rec = m.ply_vertex_records(p, c, normals=nrm)
    assert rec.shape == (5000, 51)
    assert rec.tobytes() == N.ply_normal_records(p, nrm, c).tobytes()
    # without normals: the 27-byte records of today
    assert m.ply_vertex_records(p, c).tobytes() == O.ply_records(p, c).tobytes()
    monkeypatch.chdir(tmp_path)
    (tmp_path / "outputs").mkdir()
    path = m.save_ply(p, c, "withn", normals=nrm)
    data = open(path, "rb").read()
    assert data == N.PLY_NORMAL_HEADER.format(n=5000).encode() + N.ply_normal_records(p, nrm, c).tobytes()


def test_point_cloud_stage_with_normals_equals_chained_calls(m, tmp_path, monkeypatch):
    rng = np.random.default_rng(70)
    img = rng.integers(0, 256, (240, 320, 3), dtype=np.uint8)
    dep = cases.make_depth(259, 343, 5, "scene")
    base = m.point_cloud_stage(img, dep, density="medium")
    out = m.point_cloud_stage(img, dep, density="medium", normals=True)
    for key in ("point_count", "preview_points", "preview_colors", "bounds"):
        assert out[key] == base[key]
    assert out["points"].tobytes() == base["points"].tobytes() and out["colors"].tobytes() == base["colors"].tobytes()
    assert "normals" not in base
    # by hand: stage -> refine_point_cloud -> estimate_normals -> save_ply
    p, c = m.depth_to_point_cloud(img, dep, density="medium")
    p, c = m.refine_point_cloud(p, c)
    nrm = m.estimate_normals(p)
    assert out["normals"].tobytes() == nrm.tobytes()
    monkeypatch.chdir(tmp_path)
    (tmp_path / "outputs").mkdir()
    with open(m.save_ply(p, c, "byhand", normals=nrm), "rb") as f:
        assert out["file_bytes"] == f.read()
    # the file path variant writes the same bytes
    res = m.point_cloud_stage(img, dep, density="medium", normals=True, filename="staged", return_arrays=False)
    assert open(res["filepath"], "rb").read() == out["file_bytes"] and "normals" not in res
    # other formats ignore the normals
    for fmt in ("las", "xyz"):
        a = m.point_cloud_stage(img, dep, density="medium", output_format=fmt)
        b = m.point_cloud_stage(img, dep, density="medium", output_format=fmt, normals=True)
        assert a["file_bytes"] == b["file_bytes"]
