"""GPU (-m gpu): mesh simplification (simplify_mesh, point_cloud_stage(mesh_preview_voxel=...)) against the oracle
(oracle/d2pc_simplify_oracle.py) with the bounds of tests/simplify_cases.py: counts, vertex order, vertex rows,
triangles and integral colours exact; positions and normals within the fixed-point bounds."""
import os

import numpy as np
import pytest

from oracle import d2pc_mesh_oracle as MO
from oracle import d2pc_simplify_oracle as SO
from tests import cases
from tests.simplify_cases import compare, soup
from tests.test_mesh_gpu import oracle_chain, stage_lattice
from tests.test_simplify_cpu import cube_corner, lattice_mesh

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def m():
    import torch
    assert torch.cuda.is_available()
    import image_to_pointcloud_b200 as mod
    mod.load_library()
    return mod


def run(m, mesh, vs, contraction, what=""):
    got = m.simplify_mesh(mesh, vs, contraction=contraction)
    return compare(got, mesh, vs, contraction, what)


@pytest.mark.parametrize("kind", ["uniform", "scene", "ties"])
@pytest.mark.parametrize("density", ["high", "medium"])
def test_stage_lattices(m, kind, density):
    _, _, xyz, rgb, shape = stage_lattice(97, 151, 3, kind, density)
    keep = np.random.default_rng(11).random(len(xyz)) < 0.85
    for mesh in (MO.grid_mesh(xyz, rgb, shape), MO.grid_mesh(xyz, rgb, shape, keep=keep, compute_normals=False)):
        for vs in (0.003, 0.02, 0.1):
            for c in SO.CONTRACTIONS:
                run(m, mesh, vs, c, f"{kind} {density} {vs} {c}")


def test_hand_meshes_and_soups(m):
    cube = cube_corner()
    for c in SO.CONTRACTIONS:
        run(m, cube, 0.6, c, "cube")
    got = m.simplify_mesh(cube, 0.6, contraction="quadric")
    assert np.array_equal(got.vertices[0], np.array([1.25, -0.5, 2.0], np.float32))
    rng = np.random.default_rng(3)
    xy = rng.random((300, 2)) * 2
    from scipy.spatial import Delaunay
    plane = MO.Mesh(np.concatenate([xy, np.full((300, 1), 0.75)], axis=1).astype(np.float32),
                    rng.integers(0, 256, (300, 3)).astype(np.float32), Delaunay(xy).simplices.astype(np.int32), None,
                    np.arange(300, dtype=np.int64))
    got = m.simplify_mesh(plane, 0.4, contraction="quadric")
    assert (got.vertices[:, 2] == np.float32(0.75)).all()
    run(m, plane, 0.4, "quadric", "plane")
    rot = MO.Mesh(np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [5, 5, 5]], np.float32), np.zeros((4, 3), np.float32),
                  np.array([[1, 2, 0], [0, 1, 2], [2, 0, 1], [0, 2, 1], [3, 1, 2], [1, 2, 3]], np.int32), None,
                  np.arange(4, dtype=np.int64))
    assert m.simplify_mesh(rot, 0.01).triangles.tolist() == [[0, 1, 2], [0, 2, 1], [1, 2, 3]]
    for it in range(20):
        mesh = soup(rng, int(rng.integers(1, 3000)), int(rng.integers(0, 6000)), normals=bool(it % 2),
                    integral=bool(it % 3))
        ext = float(np.ptp(mesh.vertices.astype(np.float64), axis=0).max()) or 1.0
        for f in (1e-3, 0.05, 0.3):
            for c in SO.CONTRACTIONS:
                run(m, mesh, ext * f, c, f"soup {it} {f} {c}")


def test_voxel_size_sweep(m):
    _, _, xyz, rgb, shape = stage_lattice(120, 160, 8, "scene", "high")
    mesh = MO.grid_mesh(xyz, rgb, shape)
    ext = float(np.ptp(mesh.vertices.astype(np.float64), axis=0).max())
    for vs in (1e-4, 1e-3, 0.01, 0.1, 1.0, ext, 10 * ext):
        for c in SO.CONTRACTIONS:
            run(m, mesh, vs, c, f"{vs} {c}")
    one = m.simplify_mesh(mesh, 10 * ext)
    assert len(one.vertices) == 1 and len(one.triangles) == 0


def test_index_limit(m):
    def two(x):
        return MO.Mesh(np.array([[0, 0, 0], [x, 0, 0]], np.float32), np.zeros((2, 3), np.float32),
                       np.zeros((0, 3), np.int32), None, np.arange(2, dtype=np.int64))
    ok = two(2097150.75)          # floor((x + 0.5) / 1) = 2^21 - 1
    assert SO.cluster_index(ok.vertices, 1.0)[0].max() == 2 ** 21 - 1
    got = m.simplify_mesh(ok, 1.0)
    compare(got, ok, 1.0, "average", "2^21 - 1")
    with pytest.raises(ValueError, match="too small"):
        m.simplify_mesh(two(2097151.75), 1.0)   # index 2^21
    with pytest.raises(ValueError, match="too small"):
        SO.simplify_mesh(two(2097151.75), 1.0)


def test_refused_meshes(m):
    rng = np.random.default_rng(4)
    mesh = soup(rng, 50, 80)
    bad = mesh._replace(triangles=np.concatenate([mesh.triangles, [[0, 1, 50]]]).astype(np.int32))
    with pytest.raises(ValueError, match="triangle"):
        m.simplify_mesh(bad, 0.5)
    neg = mesh._replace(triangles=np.concatenate([mesh.triangles, [[-1, 1, 2]]]).astype(np.int32))
    with pytest.raises(ValueError, match="triangle"):
        m.simplify_mesh(neg, 0.5)
    for field, k in (("vertices", 1), ("colors", 2), ("vertex_normals", 0)):
        a = getattr(mesh, field).copy()
        a[7, k] = np.nan
        with pytest.raises(ValueError, match="non-finite"):
            m.simplify_mesh(mesh._replace(**{field: a}), 0.5)
    a = mesh.vertices.copy()
    a[3, 0] = np.inf
    with pytest.raises(ValueError, match="non-finite"):
        m.simplify_mesh(mesh._replace(vertices=a), 0.5)


def test_empty_and_singleton_meshes(m):
    empty = MO.Mesh(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int32), None,
                    np.zeros(0, np.int64))
    for c in SO.CONTRACTIONS:
        got = m.simplify_mesh(empty, 0.1, contraction=c)
        assert all(len(a) == 0 for a in got if a is not None)
    with pytest.raises(ValueError, match="triangle"):
        m.simplify_mesh(empty._replace(triangles=np.zeros((1, 3), np.int32)), 0.1)
    rng = np.random.default_rng(5)
    pts = soup(rng, 400, 0)                       # T = 0
    for c in SO.CONTRACTIONS:
        run(m, pts, 0.2, c, "no triangles")
    mesh = lattice_mesh(4, normals=False)
    assert len(SO.simplify_mesh(mesh, 1e-5).vertices) == len(mesh.vertices)
    got = m.simplify_mesh(mesh, 1e-5)             # every cluster one vertex
    compare(got, mesh, 1e-5, "average", "singletons")
    assert np.array_equal(got.triangles, mesh.triangles) and np.array_equal(got.colors, mesh.colors)
    assert np.array_equal(got.vertex_rows, mesh.vertex_rows)


def test_full_1080p_high_frame_through_depth_to_mesh(m):
    img, dep = cases.make_image(1080, 1920, 1), cases.make_depth(1080, 1920, 1, "scene")
    mesh = m.depth_to_mesh(img, dep, "high")
    assert len(mesh.vertices) > 1_000_000
    for vs, c in ((0.01, "average"), (0.02, "quadric")):
        stats = run(m, mesh, vs, c, f"1080p {vs} {c}")
        assert stats["clusters"] > 1000


def test_device_tensors_and_repeatability(m):
    import torch
    _, _, xyz, rgb, shape = stage_lattice(101, 133, 7, "scene", "high")
    mesh = MO.grid_mesh(xyz, rgb, shape)
    dev = m.TriangleMesh(*(torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in mesh))
    for c in SO.CONTRACTIONS:
        host = m.simplify_mesh(mesh, 0.02, contraction=c)
        again = m.simplify_mesh(mesh, 0.02, contraction=c)
        on_dev = m.simplify_mesh(dev, 0.02, contraction=c, return_device=True)
        assert all(t.is_cuda for t in on_dev)
        for a, b, d in zip(host, again, on_dev):
            assert a.tobytes() == b.tobytes() == d.cpu().numpy().tobytes()
        assert m.mesh_ply_bytes(on_dev) == m.mesh_ply_bytes(host)


def test_point_cloud_stage_mesh_preview(m, tmp_path):
    img, dep = cases.make_image(80, 120, 4), cases.make_depth(80, 120, 4, "scene")
    base = m.point_cloud_stage(img, dep, density="high", mesh=True)
    out = m.point_cloud_stage(img, dep, density="high", mesh=True, mesh_preview_voxel=0.05)
    for k, v in base.items():   # every other output is unchanged
        if isinstance(v, np.ndarray):
            assert v.tobytes() == out[k].tobytes(), k
        else:
            assert v == out[k], k
    full = oracle_chain(img, dep, "high", refine=True)
    chained = m.simplify_mesh(m.depth_to_mesh(img, dep, "high", refine=True), 0.05)
    compare(chained, full, 0.05, "average", "stage chain")
    assert out["mesh_preview_vertex_count"] == len(chained.vertices)
    assert out["mesh_preview_triangle_count"] == len(chained.triangles)
    assert out["mesh_preview_file_bytes"] == m.mesh_ply_bytes(chained)
    want = SO.simplify_mesh(full, 0.05)
    assert len(out["mesh_preview_file_bytes"]) == len(MO.mesh_ply_bytes(want))
    cwd = os.getcwd()
    try:
        os.chdir(tmp_path)
        f = m.point_cloud_stage(img, dep, density="high", mesh=True, mesh_preview_voxel=0.05, filename="scene",
                                return_arrays=False)
        assert f["mesh_preview_filepath"] == "outputs/scene_mesh_preview.ply"
        assert open(f["mesh_preview_filepath"], "rb").read() == out["mesh_preview_file_bytes"]
    finally:
        os.chdir(cwd)
