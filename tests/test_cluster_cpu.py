"""CPU: the density-clustering oracle (oracle/d2pc_cluster_oracle.py).  Its vectorised DBSCAN equals the restatement
of Open3D's loop, and its radius outlier removal equals brute force, on random small clouds; hand cases pin the
labels; the argument checks of the oracle and of the package agree."""
import numpy as np
import pytest

from oracle import d2pc_cluster_oracle as CL


def cloud(kind, rng, n=160):
    if kind == "uniform":
        p = rng.random((n, 3))
    elif kind == "blobs":
        c = rng.random((4, 3))
        p = c[rng.integers(0, 4, n)] + rng.normal(0, 0.03, (n, 3))
    elif kind == "lines":
        t = rng.random(n)
        p = np.stack([t, 0.5 * t, np.where(rng.random(n) < 0.5, 0.0, 0.3)], 1) + rng.normal(0, 0.002, (n, 3))
    elif kind == "planes":
        p = rng.random((n, 3))
        p[:, 2] = np.round(p[:, 2] * 3) / 3
    elif kind == "duplicates":
        p = np.repeat(rng.random((n // 8, 3)), 8, axis=0)
    elif kind == "lattice":
        g = np.arange(6) * 0.05
        p = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)[:n]
    elif kind == "clump":   # pixels clipped at a percentile: one tiny lattice, plus a surface
        p = rng.random((n, 3))
        k = n // 3
        p[:k] = 0.4 + rng.integers(0, 4, (k, 3)) * 1e-7
    return np.ascontiguousarray(p, dtype=np.float32)


KINDS = ["uniform", "blobs", "lines", "planes", "duplicates", "lattice", "clump"]


@pytest.mark.parametrize("kind", KINDS)
def test_vectorised_equals_open3d_loop(kind):
    rng = np.random.default_rng(KINDS.index(kind))
    for trial in range(6):
        p = cloud(kind, rng)
        eps = float(rng.choice([0.02, 0.05, 0.08, 0.15]))
        for min_points in (0, 1, 2, 3, 5, 10, 30):
            want = CL.cluster_dbscan_loop(p, eps, min_points)
            got = CL.cluster_dbscan(p, eps, min_points)
            assert got.dtype == np.int32 and np.array_equal(got, want), (kind, trial, eps, min_points)


@pytest.mark.parametrize("kind", KINDS)
def test_radius_outlier_equals_brute_force(kind):
    rng = np.random.default_rng(100 + KINDS.index(kind))
    for trial in range(4):
        p = cloud(kind, rng)
        r = float(rng.choice([0.03, 0.07, 0.12]))
        for nb in (1, 2, 4, 9, 20):
            assert np.array_equal(CL.remove_radius_outlier(p, nb, r), CL.remove_radius_outlier_brute(p, nb, r))


def f32(rows):
    return np.asarray(rows, dtype=np.float32)


def test_chain_linked_through_cores():
    p = f32([[0.1 * k, 0, 0] for k in range(10)])
    assert CL.cluster_dbscan(p, 0.15, 3).tolist() == [0] * 10   # the ends are border points of the one chain
    assert CL.cluster_dbscan(p, 0.15, 4).tolist() == [-1] * 10


def test_border_point_takes_the_lower_cluster():
    a = [[-0.01 * k, 0, 0] for k in range(4)]
    b = [[1.0 + 0.01 * k, 0, 0] for k in range(4)]
    mid = [[0.5, 0, 0]]     # within eps of a[0] and b[0] only: not core
    p = f32(b + mid + a)    # cluster 0 is b (lowest core index), cluster 1 is a
    lab = CL.cluster_dbscan(p, 0.505, 4)
    assert lab.tolist() == [0, 0, 0, 0, 0, 1, 1, 1, 1]
    assert np.array_equal(lab, CL.cluster_dbscan_loop(p, 0.505, 4))
    p = f32(a + mid + b)
    assert CL.cluster_dbscan(p, 0.505, 4).tolist() == [0, 0, 0, 0, 0, 1, 1, 1, 1]


def test_noise_first_absorbed_later():
    # row 0 is visited first, is not core, and becomes a border point of the cluster seeded later
    p = f32([[0.0, 0, 0], [0.09, 0, 0], [0.1, 0, 0], [0.11, 0, 0], [0.1, 0.01, 0]])
    lab = CL.cluster_dbscan(p, 0.095, 4)
    assert lab.tolist() == [0, 0, 0, 0, 0]
    assert np.array_equal(lab, CL.cluster_dbscan_loop(p, 0.095, 4))


def test_isolated_points_min_points_one():
    p = f32([[0, 0, 0], [1, 0, 0], [2, 0, 0]])
    assert CL.cluster_dbscan(p, 0.5, 1).tolist() == [0, 1, 2]
    assert CL.cluster_dbscan(p, 0.5, 0).tolist() == [0, 1, 2]
    assert CL.cluster_dbscan(p, 0.5, 2).tolist() == [-1, -1, -1]


def test_exact_eps_is_not_a_neighbour():
    eps = 0.25                               # d2 == eps * eps exactly: not neighbours (strict)
    p = f32([[0, 0, 0], [0.25, 0, 0]])
    assert CL.cluster_dbscan(p, eps, 2).tolist() == [-1, -1]
    below = np.nextafter(np.float32(0.25), np.float32(0))   # one ulp closer: neighbours
    p = f32([[0, 0, 0], [below, 0, 0]])
    assert CL.cluster_dbscan(p, eps, 2).tolist() == [0, 0]
    assert CL.remove_radius_outlier(p, 1, eps).tolist() == [0, 1]
    assert CL.remove_radius_outlier(f32([[0, 0, 0], [0.25, 0, 0]]), 1, eps).tolist() == []


def test_remove_small_clusters():
    p = f32([[0, 0, 0], [0.01, 0, 0], [0.02, 0, 0], [5, 5, 5], [5.01, 5, 5], [9, 9, 9]])
    kept, lab, sizes = CL.remove_small_clusters(p, 0.05, 2, min_size=3)
    assert lab.tolist() == [0, 0, 0, 1, 1, -1] and sizes.tolist() == [3, 2] and kept.tolist() == [0, 1, 2]
    assert CL.remove_small_clusters(p, 0.05, 2)[0].tolist() == [0, 1, 2, 3, 4]


def test_refusals_and_empty():
    import image_to_pointcloud_b200.cluster as C
    p = f32([[0, 0, 0], [1, 0, 0]])
    for bad in (0.0, -1.0, float("nan"), float("inf"), 1e-200):
        with pytest.raises(ValueError):
            CL.cluster_dbscan(p, bad, 2)
        with pytest.raises(ValueError):
            C.cluster_dbscan(p, bad, 2)
    for bad in (-1, 2.5):
        with pytest.raises(ValueError):
            CL.cluster_dbscan(p, 0.1, bad)
        with pytest.raises(ValueError):
            C.cluster_dbscan(p, 0.1, bad)
    with pytest.raises(ValueError, match="finite"):
        CL.cluster_dbscan(f32([[0, 0, np.nan]]), 0.1, 2)
    with pytest.raises(ValueError, match="finite"):
        C.cluster_dbscan(f32([[0, 0, np.inf]]), 0.1, 2)
    for nb, r in ((0, 0.1), (2, 0.0), (2, float("nan"))):
        with pytest.raises(ValueError, match="number of points and radius must be positive"):
            CL.remove_radius_outlier(p, nb, r)
        with pytest.raises(ValueError, match="number of points and radius must be positive"):
            C.remove_radius_outlier(p, nb_points=nb, radius=r)
    with pytest.raises(ValueError):
        C.remove_small_clusters(p, eps=0.1, min_points=2, min_size=0)
    assert CL.cluster_dbscan(np.zeros((0, 3), np.float32), 0.1, 2).shape == (0,)


def test_grid_limit():
    # extent 1 along x: eps / 2 cells fit while 1 / cs < 1048574
    p = f32([[0, 0, 0], [1, 0, 0]])
    cs_ok = 1.0 / 1048573.0
    eps_ok = cs_ok / (0.5 * (1 + 2.0 ** -20))
    assert CL.grid_fits(p, eps_ok)
    assert CL.cluster_dbscan(p, eps_ok, 1).tolist() == [0, 1]
    eps_bad = (1.0 / 1048574.0) / (0.5 * (1 + 2.0 ** -20))
    assert not CL.grid_fits(p, eps_bad)
    import image_to_pointcloud_b200.cluster as C
    with pytest.raises(ValueError, match="too small"):
        CL.cluster_dbscan(p, eps_bad, 1)
    with pytest.raises(ValueError, match="too small"):
        C.cluster_dbscan(p, eps_bad, 1)
    with pytest.raises(ValueError, match="too small"):
        C.remove_small_clusters(p, eps=eps_bad, min_points=1)
    # a single point, or coincident points, fit at any eps
    assert CL.grid_fits(f32([[3, 3, 3]] * 4), 1e-30)
