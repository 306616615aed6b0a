"""GPU (-m gpu): density clustering (cluster_dbscan, remove_radius_outlier, remove_small_clusters,
point_cloud_stage(cluster_eps=...)) against the oracle (oracle/d2pc_cluster_oracle.py), bit for bit."""
import numpy as np
import pytest

from oracle import d2pc_cluster_oracle as CL
from oracle import d2pc_mesh_oracle as MO
from oracle import d2pc_oracle as O
from tests import cases
from tests.test_mesh_gpu import stage_lattice

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def m():
    import torch
    assert torch.cuda.is_available()
    import image_to_pointcloud_b200 as mod
    mod.load_library()
    return mod


def median_spacing(p):
    from scipy.spatial import cKDTree
    d, _ = cKDTree(p.astype(np.float64)).query(p.astype(np.float64), k=2)
    return float(np.median(d[:, 1]))


def check_all(m, p, eps, min_points, min_size=1, rgb=None, nb_points=None, what=""):
    """labels, kept rows and kept indices of the device equal the oracle's; returns the labels"""
    want = CL.cluster_dbscan(p, eps, min_points)
    got = m.cluster_dbscan(p, eps, min_points)
    assert got.dtype == np.int32 and got.shape == want.shape, what
    if not np.array_equal(got, want):
        raise AssertionError(f"{what}: {(got != want).sum()} of {len(p)} labels differ")
    kidx, _, sizes = CL.remove_small_clusters(p, eps, min_points, min_size)
    gp, gc, gi = m.remove_small_clusters(p, rgb, eps=eps, min_points=min_points, min_size=min_size)
    assert np.array_equal(gi, kidx), what
    assert gp.tobytes() == p[kidx].tobytes(), what
    assert (gc is None) if rgb is None else gc.tobytes() == rgb[kidx].tobytes(), what
    if nb_points is not None:
        want_r = CL.remove_radius_outlier(p, nb_points, eps)
        rp, _, ri = m.remove_radius_outlier(p, nb_points=nb_points, radius=eps)
        assert np.array_equal(ri, want_r) and rp.tobytes() == p[want_r].tobytes(), what
    return got


@pytest.mark.parametrize("kind", ["uniform", "scene", "ties"])
@pytest.mark.parametrize("density", ["high", "medium"])
def test_stage_clouds(m, kind, density):
    _, _, xyz, rgb, _ = stage_lattice(97, 151, 3, kind, density)
    sor, _, _ = O.statistical_outlier_removal(xyz)
    for name, p, c in (("raw", xyz, rgb), ("sor", xyz[sor], rgb[sor])):
        h = median_spacing(p)
        for f in (2.0, 5.0):
            for min_points, min_size in ((10, 1), (4, 25)):
                check_all(m, p, f * h, min_points, min_size, rgb=c, nb_points=min_points,
                          what=f"{kind} {density} {name} {f} {min_points}")


def test_cell_faces_and_ulp_pairs(m):
    rng = np.random.default_rng(5)
    eps = 0.1
    cs = CL.cell_size(eps)
    k = rng.integers(0, 40, (3000, 3))
    faces = (k * cs).astype(np.float32)                      # on (rounded) cell faces
    # pairs one ulp either side of eps along x, each pair far (>= 1) from every other one
    g = np.stack(np.meshgrid(*[np.arange(12.0)] * 3, indexing="ij"), -1).reshape(-1, 3)
    a = (g + rng.random(g.shape) * 0.5).astype(np.float32)
    b = a.copy()
    b[:, 0] = a[:, 0] + np.float32(0.25)
    e = float(b[0, 0]) - float(a[0, 0])
    pairs = []
    for t in range(len(a)):
        if float(b[t, 0]) - float(a[t, 0]) != e:
            continue
        bx = (b[t, 0], np.nextafter(b[t, 0], np.float32(-1)), np.nextafter(b[t, 0], np.float32(99)))[t % 3]
        pairs += [a[t], [bx, a[t, 1], a[t, 2]]]
    p = np.concatenate([faces, np.asarray(pairs, np.float32)]).astype(np.float32)
    check_all(m, faces, eps, 2, nb_points=2, what="faces")
    check_all(m, faces, eps, 9, nb_points=6, what="faces 9")
    lab = check_all(m, np.asarray(pairs, np.float32), e, 2, nb_points=1, what="ulp pairs")
    assert (lab >= 0).any() and (lab < 0).any()
    check_all(m, p, e, 3, what="both")


def test_one_cell_of_a_million(m):
    p = np.tile(np.float32([[1.5, -2.0, 3.25]]), (1_000_000, 1))
    lab = m.cluster_dbscan(p, 0.01, 10)
    assert (lab == 0).all()
    _, _, idx = m.remove_small_clusters(p, eps=0.01, min_points=1_000_000, min_size=1_000_000)
    assert np.array_equal(idx, np.arange(1_000_000))
    _, _, idx = m.remove_small_clusters(p, eps=0.01, min_points=1_000_001)
    assert len(idx) == 0
    _, _, idx = m.remove_radius_outlier(p, nb_points=999_999, radius=0.01)
    assert len(idx) == 1_000_000


def test_a_million_isolated(m):
    g = np.arange(100, dtype=np.float32)
    p = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    p = p[np.random.default_rng(2).permutation(len(p))]
    assert (m.cluster_dbscan(p, 0.5, 2) == -1).all()
    assert np.array_equal(m.cluster_dbscan(p, 0.5, 1), np.arange(len(p), dtype=np.int32))
    check_all(m, p[:200_000], 1.01, 2, what="lattice")


def test_a_chain_of_a_million(m):
    n = 1_000_000
    t = np.arange(n, dtype=np.float64)
    p = np.stack([np.cos(t * 1e-4) * 60.0, np.sin(t * 1e-4) * 60.0, t * 1e-5], 1).astype(np.float32)
    p = p[np.random.default_rng(3).permutation(n)]
    lab = check_all(m, p, 0.01, 2, what="chain")
    assert (lab == 0).all()


def test_1080p_medium_frame(m):
    img, dep = cases.make_image(1080, 1920, 0), cases.make_depth(1080, 1920, 0, "scene")
    xyz, rgb = O.depth_to_point_cloud(img, dep, density="medium")
    p, c, _, _ = m.statistical_outlier_removal(xyz, rgb)
    h = median_spacing(p)
    check_all(m, p, 2.0 * h, 10, min_size=50, rgb=c, nb_points=10, what="1080p medium")


def test_refusals(m):
    import torch
    p = np.random.default_rng(0).random((100, 3)).astype(np.float32)
    bad = p.copy()
    bad[7, 1] = np.nan
    for fn in (lambda q, e: m.cluster_dbscan(q, e, 3), lambda q, e: m.remove_small_clusters(q, eps=e, min_points=3),
               lambda q, e: m.remove_radius_outlier(q, nb_points=3, radius=e)):
        with pytest.raises(ValueError, match="finite"):
            fn(bad, 0.1)
        with pytest.raises(ValueError, match="finite"):
            fn(torch.from_numpy(bad).cuda(), 0.1)      # device rows: the kernels' error word
        with pytest.raises(ValueError, match="too small"):
            fn(p, 1e-7)
        with pytest.raises(ValueError, match="too small"):
            fn(torch.from_numpy(p).cuda(), 1e-7)
        for e in (0.0, -1.0, float("nan"), float("inf")):
            with pytest.raises(ValueError):
                fn(p, e)
    with pytest.raises(ValueError):
        m.cluster_dbscan(p, 0.1, -1)
    assert m.cluster_dbscan(np.zeros((0, 3), np.float32), 0.1, 3).shape == (0,)
    q, c, i = m.remove_small_clusters(np.zeros((0, 3), np.float32), eps=0.1, min_points=3)
    assert q.shape == (0, 3) and c is None and i.shape == (0,)


def test_device_tensors_and_repeat(m):
    import torch
    _, _, xyz, rgb, _ = stage_lattice(120, 160, 9, "scene", "high")
    eps = 3.0 * median_spacing(xyz)
    want = CL.cluster_dbscan(xyz, eps, 10)
    lab = m.cluster_dbscan(torch.from_numpy(xyz).cuda(), eps, 10, return_device=True)
    assert lab.is_cuda and lab.dtype == torch.int32 and np.array_equal(lab.cpu().numpy(), want)
    kidx, _, _ = CL.remove_small_clusters(xyz, eps, 10, 5)
    dp, dc, di = m.remove_small_clusters(torch.from_numpy(xyz).cuda(), torch.from_numpy(rgb).cuda(), eps=eps,
                                         min_points=10, min_size=5, return_device=True)
    assert dp.is_cuda and dc.is_cuda and di.is_cuda
    assert np.array_equal(di.cpu().numpy(), kidx) and dc.cpu().numpy().tobytes() == rgb[kidx].tobytes()
    runs = [(m.cluster_dbscan(xyz, eps, 10), m.remove_small_clusters(xyz, rgb, eps=eps, min_points=10, min_size=5),
             m.remove_radius_outlier(xyz, rgb, nb_points=10, radius=eps)) for _ in range(2)]
    a, b = runs
    assert a[0].tobytes() == b[0].tobytes()
    for x, y in zip(a[1] + a[2], b[1] + b[2]):
        assert x.tobytes() == y.tobytes()


def test_stage(m):
    img, dep = cases.make_image(80, 120, 4), cases.make_depth(80, 120, 4, "scene")
    base = m.point_cloud_stage(img, dep, density="high", mesh=True)
    off = m.point_cloud_stage(img, dep, density="high", mesh=True, cluster_eps=None)
    assert base.keys() == off.keys()
    for k, v in base.items():   # the knob left at None changes nothing
        assert (v.tobytes() == off[k].tobytes()) if isinstance(v, np.ndarray) else v == off[k], k
    xyz, rgb = O.depth_to_point_cloud(img, dep, density="high")
    sor, _, _ = O.statistical_outlier_removal(xyz)
    eps = 3.0 * median_spacing(xyz[sor])
    out = m.point_cloud_stage(img, dep, density="high", mesh=True, cluster_eps=eps, cluster_min_points=10,
                              cluster_min_size=40)
    kidx, labels, _ = CL.remove_small_clusters(xyz[sor], eps, 10, 40)
    rows = sor[kidx]
    pts, cols = xyz[rows], rgb[rows]
    assert out["cluster_count"] == int(labels.max()) + 1
    assert out["cluster_removed_point_count"] == len(sor) - len(rows) > 0
    assert out["point_count"] == len(rows)
    assert out["points"].tobytes() == pts.tobytes() and out["colors"].tobytes() == cols.tobytes()
    pp, pc = O.preview_rows(pts, cols)
    assert out["preview_points"] == pp.astype(float).tolist() and out["preview_colors"] == pc.astype(float).tolist()
    from image_to_pointcloud_b200 import writers
    head = writers.PLY_HEADER.format(n=len(rows)).encode("ascii")
    assert out["file_bytes"] == head + O.ply_records(pts, cols).tobytes()
    b = out["bounds"]
    assert [b["minX"], b["minY"], b["minZ"]] == [float(v) for v in pts.min(0)]
    assert [b["maxX"], b["maxY"], b["maxZ"]] == [float(v) for v in pts.max(0)]
    keep = np.zeros(len(xyz), bool)
    keep[rows] = True
    st = O.DENSITY_STEP["high"]
    want = MO.grid_mesh(xyz, rgb, (-(-80 // st), -(-120 // st)), keep=keep)
    assert out["mesh_file_bytes"] == MO.mesh_ply_bytes(want)
    with pytest.raises(ValueError):
        m.point_cloud_stage(img, dep, cluster_eps=-1.0)
    with pytest.raises(ValueError):
        m.point_cloud_stage(img, dep, cluster_eps=0.1, cluster_min_size=0)
