"""GPU (-m gpu): the lattice mesh (grid_mesh, depth_to_mesh, point_cloud_stage(mesh=True), the mesh PLY) against the
oracle's restatement (oracle/d2pc_mesh_oracle.py), bit for bit: float32 words of vertices and colours, int32
triangles, vertex rows and float64 words of the normals."""
import os

import numpy as np
import pytest

from oracle import d2pc_mesh_oracle as MO
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


def assert_same(got, want, what=""):
    for f in MO.Mesh._fields:
        g, w = getattr(got, f), getattr(want, f)
        if g is None or w is None:
            assert g is None and w is None, f"{what}: {f}"
            continue
        g = np.ascontiguousarray(g)
        assert g.shape == w.shape and g.dtype == w.dtype, f"{what}: {f} {g.shape}/{g.dtype} != {w.shape}/{w.dtype}"
        if g.tobytes() != w.tobytes():
            bad = (g.reshape(len(g), -1) != w.reshape(len(w), -1)).any(axis=1).sum() if len(g) else 0
            raise AssertionError(f"{what}: {f}: {bad} of {len(g)} rows differ")


def check(m, xyz, rgb, shape, **kw):
    want = MO.grid_mesh(xyz, rgb, shape, **kw)
    got = m.grid_mesh(xyz, rgb, shape, **kw)
    assert_same(got, want, f"{shape} {kw.get('max_edge')} {kw.get('max_angle')}")
    return got


def stage_lattice(H, W, seed, kind, density, invert=True):
    img = cases.make_image(H, W, seed)
    dep = cases.make_depth(H, W, seed, kind)
    xyz, rgb = O.depth_to_point_cloud(img, dep, density=density, invert=invert)
    s = O.DENSITY_STEP[density]
    return img, dep, xyz, rgb, (-(-H // s), -(-W // s))


@pytest.mark.parametrize("kind", ["uniform", "scene", "ties"])
@pytest.mark.parametrize("density", ["high", "medium"])
def test_stage_lattices_bit_exact(m, kind, density):
    _, _, xyz, rgb, shape = stage_lattice(97, 151, 3, kind, density)
    rng = np.random.default_rng(11)
    keep = rng.random(len(xyz)) < 0.85
    check(m, xyz, rgb, shape)
    check(m, xyz, rgb, shape, keep=keep, max_edge=0.05, max_angle=80.0)
    check(m, xyz, rgb, shape, keep=keep, remove_unreferenced=False, compute_normals=False)
    check(m, xyz, rgb, shape, max_angle=90.0, remove_unreferenced=False)


@pytest.mark.parametrize("shape", [(1, 1), (1, 300), (300, 1), (2, 2), (5, 127), (5, 128), (5, 129), (3, 257),
                                   (130, 3)])
def test_odd_lattice_shapes(m, shape):
    rng = np.random.default_rng(shape[0] * 1000 + shape[1])
    R, Cc = shape
    z = rng.random((R, Cc)) * 2 + 1
    z[rng.random((R, Cc)) < 0.1] += 5
    v, u = np.mgrid[0:R, 0:Cc].astype(np.float64)
    xyz = np.stack([(u - Cc / 2) * z / 300, (v - R / 2) * z / 300, z], -1).reshape(-1, 3).astype(np.float32)
    xyz[rng.random(R * Cc) < 0.05] = np.nan
    rgb = rng.integers(0, 256, (R * Cc, 3)).astype(np.float32)
    for kw in (dict(), dict(keep=rng.random(R * Cc) < 0.8, max_edge=0.02), dict(remove_unreferenced=False)):
        check(m, xyz, rgb, shape, **kw)


def test_full_1080p_high_frame(m):
    _, _, xyz, rgb, shape = stage_lattice(1080, 1920, 1, "scene", "high")
    got = check(m, xyz, rgb, shape)
    assert len(got.triangles) > 0 and len(got.vertices) > 0


def test_clipped_percentile_apex(m):
    # with invert, the pixels clipped at the 98th percentile sit ~5e-7 from the camera (z = 5.2e-7 here):
    # near-degenerate triangles between them and between them and their neighbours
    _, _, xyz, rgb, shape = stage_lattice(120, 160, 5, "uniform", "high", invert=True)
    apex = np.abs(xyz[:, 2]) < 1e-5
    assert apex.sum() > 100 and np.abs(xyz[apex]).max() < 1e-5
    check(m, xyz, rgb, shape, max_angle=90.0)
    check(m, xyz, rgb, shape, max_angle=90.0, remove_unreferenced=False, max_edge=1e-6)


def test_device_tensors_and_repeatability(m):
    import torch
    _, _, xyz, rgb, shape = stage_lattice(101, 133, 7, "scene", "high")
    keep = np.random.default_rng(1).random(len(xyz)) < 0.9
    want = MO.grid_mesh(xyz, rgb, shape, keep=keep)
    dx, dr, dk = (torch.from_numpy(a).cuda() for a in (xyz, rgb, keep))
    got = m.grid_mesh(dx, dr, shape, keep=dk, return_device=True)
    assert all(t.is_cuda for t in got if t is not None)
    assert got.vertex_rows.dtype == torch.int64 and got.triangles.dtype == torch.int32
    assert_same(m.TriangleMesh(*(t.cpu().numpy() for t in got)), want, "device in / out")
    again = m.grid_mesh(xyz, rgb, shape, keep=keep)
    for a, b in zip(again, m.grid_mesh(xyz, rgb, shape, keep=keep)):
        assert a.tobytes() == b.tobytes()


def oracle_chain(img, dep, density, z_range=None, refine=False, **kw):
    xyz, rgb = O.depth_to_point_cloud(img, dep, density=density)
    keep = np.ones(len(xyz), bool) if z_range is None else O.range_mask(xyz, *z_range)
    if refine:
        rows = np.nonzero(keep)[0]
        kept, _, _ = O.statistical_outlier_removal(xyz[rows])
        keep = np.zeros(len(xyz), bool)
        keep[rows[kept]] = True
    s = O.DENSITY_STEP[density]
    H, W = img.shape[:2]
    return MO.grid_mesh(xyz, rgb, (-(-H // s), -(-W // s)), keep=keep, **kw)


@pytest.mark.parametrize("z_range,refine", [(None, False), ((3.0, 9.0), False), ((2.0, 9.5), True), (None, True)])
def test_depth_to_mesh_equals_oracle_chain(m, z_range, refine):
    img, dep = cases.make_image(90, 140, 2), cases.make_depth(97, 151, 2, "scene")
    got = m.depth_to_mesh(img, dep, "medium", z_range=z_range, refine=refine, max_edge=0.3)
    assert_same(got, oracle_chain(img, dep, "medium", z_range, refine, max_edge=0.3), f"{z_range} {refine}")


def test_point_cloud_stage_mesh(m, tmp_path):
    img, dep = cases.make_image(80, 120, 4), cases.make_depth(80, 120, 4, "scene")
    base = m.point_cloud_stage(img, dep, density="high")
    out = m.point_cloud_stage(img, dep, density="high", mesh=True, mesh_max_angle=80.0)
    for k, v in base.items():   # every point-cloud output is unchanged
        if isinstance(v, np.ndarray):
            assert v.tobytes() == out[k].tobytes(), k
        else:
            assert v == out[k], k
    want = oracle_chain(img, dep, "high", refine=True, max_angle=80.0)
    assert out["mesh_vertex_count"] == len(want.vertices) and out["mesh_triangle_count"] == len(want.triangles)
    assert out["mesh_file_bytes"] == MO.mesh_ply_bytes(want)
    chained = m.depth_to_mesh(img, dep, "high", refine=True, max_angle=80.0)
    assert m.mesh_ply_bytes(chained) == out["mesh_file_bytes"]
    cwd = os.getcwd()
    try:
        os.chdir(tmp_path)
        f = m.point_cloud_stage(img, dep, density="high", mesh=True, mesh_max_angle=80.0, filename="scene",
                                return_arrays=False)
        assert f["mesh_filepath"] == "outputs/scene_mesh.ply"
        assert open(f["mesh_filepath"], "rb").read() == MO.mesh_ply_bytes(want)
    finally:
        os.chdir(cwd)


@pytest.mark.parametrize("normals", [True, False])
def test_mesh_ply_file_equals_oracle(m, tmp_path, normals):
    _, _, xyz, rgb, shape = stage_lattice(70, 90, 9, "uniform", "high")
    keep = np.random.default_rng(2).random(len(xyz)) < 0.7
    mesh = m.grid_mesh(xyz, rgb, shape, keep=keep, compute_normals=normals, return_device=True)
    want = MO.mesh_ply_bytes(MO.grid_mesh(xyz, rgb, shape, keep=keep, compute_normals=normals))
    assert m.mesh_ply_bytes(mesh) == want
    cwd = os.getcwd()
    try:
        os.chdir(tmp_path)
        path = m.save_mesh_ply(mesh, "grid")
        assert path == "outputs/grid.ply" and open(path, "rb").read() == want
        empty = m.grid_mesh(xyz, rgb, shape, keep=np.zeros(len(xyz), bool), compute_normals=normals)
        assert open(m.save_mesh_ply(empty, "empty"), "rb").read() == MO.mesh_ply_bytes(
            MO.grid_mesh(xyz, rgb, shape, keep=np.zeros(len(xyz), bool), compute_normals=normals))
    finally:
        os.chdir(cwd)
