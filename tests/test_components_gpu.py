"""GPU (-m gpu): mesh components (cluster_connected_triangles, remove_triangles_by_mask, remove_small_components,
depth_to_mesh(min_component_triangles=...), point_cloud_stage(mesh_min_triangles=...)) against the oracle
(oracle/d2pc_components_oracle.py), bit for bit."""
import os

import numpy as np
import pytest

from oracle import d2pc_components_oracle as CO
from oracle import d2pc_mesh_oracle as MO
from oracle import d2pc_simplify_oracle as SO
from tests import cases
from tests import components_cases as CC
from tests.test_mesh_gpu import assert_same, oracle_chain, stage_lattice

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def m():
    import torch
    assert torch.cuda.is_available()
    import image_to_pointcloud_b200 as mod
    mod.load_library()
    return mod


def run(m, mesh, what=""):
    got = m.cluster_connected_triangles(mesh)
    return CC.compare(got, mesh, what)


@pytest.mark.parametrize("kind", ["uniform", "scene", "ties"])
@pytest.mark.parametrize("density", ["high", "medium"])
def test_stage_lattices(m, kind, density):
    _, _, xyz, rgb, shape = stage_lattice(97, 151, 3, kind, density)
    keep = np.random.default_rng(11).random(len(xyz)) < 0.85
    rng = np.random.default_rng(12)
    for mesh in (MO.grid_mesh(xyz, rgb, shape), MO.grid_mesh(xyz, rgb, shape, keep=keep, max_angle=70.0)):
        run(m, mesh, f"{kind} {density}")
        run(m, CC.shuffled(mesh, rng), f"{kind} {density} shuffled")
        run(m, SO.simplify_mesh(mesh, 0.02), f"{kind} {density} simplified")


def test_hand_meshes_and_soups(m):
    for name, (mesh, want) in CC.hand_meshes().items():
        got = run(m, mesh, name)
        assert got[0].tolist() == want
    rng = np.random.default_rng(3)
    for it in range(30):
        V = int(rng.integers(1, 3000))
        mesh = CC.soup(rng, V, int(rng.integers(0, 3 * V)))
        want = run(m, mesh, f"soup {it}")
        CC.check_areas(mesh, *want)


def test_union_find_stress_shapes(m):
    for what, mesh in (("strip", CC.strip(200_001)), ("comb", CC.comb(300, 200)), ("fan", CC.edge_fan(10_000)),
                       ("isolated", CC.isolated(1_000_000))):
        want = run(m, mesh, what)
        if what == "isolated":
            assert len(want[1]) == 1_000_000
        elif what != "comb":
            assert len(want[1]) == 1


def test_full_1080p_high_scene_mesh(m):
    img, dep = cases.make_image(1080, 1920, 1), cases.make_depth(1080, 1920, 1, "scene")
    mesh = m.depth_to_mesh(img, dep, "high")
    assert len(mesh.triangles) > 2_000_000
    want = run(m, mesh, "1080p high")
    CC.check_areas(mesh, *want)


def test_refused_meshes(m):
    mesh = CC.soup(np.random.default_rng(4), 50, 80)
    for bad in ([[0, 1, 50]], [[-1, 1, 2]]):
        t = np.concatenate([mesh.triangles, np.asarray(bad, np.int32)])
        with pytest.raises(ValueError, match="vertex that does not exist"):
            m.cluster_connected_triangles(mesh._replace(triangles=t))
        with pytest.raises(ValueError, match="vertex that does not exist"):
            m.remove_triangles_by_mask(mesh._replace(triangles=t), np.zeros(len(t), bool))
    v = mesh.vertices.copy()
    v[7, 1] = np.nan
    with pytest.raises(ValueError, match="non-finite"):
        m.cluster_connected_triangles(mesh._replace(vertices=v))
    with pytest.raises(ValueError, match="non-finite"):
        m.remove_small_components(mesh._replace(vertices=v), min_triangles=3)
    empty = CC.mesh_of(np.zeros((0, 3)), np.zeros((0, 3)))
    assert all(len(a) == 0 for a in m.cluster_connected_triangles(empty))
    with pytest.raises(ValueError, match="vertex that does not exist"):
        m.cluster_connected_triangles(empty._replace(triangles=np.zeros((1, 3), np.int32)))
    pts = CC.mesh_of(np.ones((5, 3)), np.zeros((0, 3)))
    assert all(len(a) == 0 for a in m.cluster_connected_triangles(pts))
    out = m.remove_triangles_by_mask(pts, np.zeros(0, bool))
    assert len(out.vertices) == 0
    out = m.remove_triangles_by_mask(pts, np.zeros(0, bool), remove_unreferenced=False)
    assert_same(out, pts._replace(vertex_normals=None), "no triangles")


def test_removal_against_the_oracle(m):
    rng = np.random.default_rng(5)
    _, _, xyz, rgb, shape = stage_lattice(97, 151, 3, "scene", "high")
    base = MO.grid_mesh(xyz, rgb, shape, max_angle=60.0)
    for mesh in (base, base._replace(vertex_normals=None), CC.soup(rng, 500, 900, normals=True)):
        T = len(mesh.triangles)
        for mask in (np.zeros(T, bool), np.ones(T, bool), rng.random(T) < 0.3, rng.random(T) < 0.9):
            for unref in (True, False):
                got = m.remove_triangles_by_mask(mesh, mask, remove_unreferenced=unref)
                assert_same(got, CO.remove_triangles_by_mask(mesh, mask, unref), f"mask {unref}")
        for kw in (dict(min_triangles=10), dict(min_triangles=1), dict(min_area=1e-3),
                   dict(min_triangles=50, min_area=1e-2)):
            assert_same(m.remove_small_components(mesh, **kw), CO.remove_small_components(mesh, **kw), f"{kw}")


def test_device_tensors_and_repeatability(m):
    import torch
    img, dep = cases.make_image(240, 320, 6), cases.make_depth(240, 320, 6, "scene")
    mesh = m.depth_to_mesh(img, dep, "high")
    dev = m.TriangleMesh(*(torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in mesh))
    a, b = m.cluster_connected_triangles(mesh), m.cluster_connected_triangles(mesh)
    d = m.cluster_connected_triangles(dev, return_device=True)
    assert all(t.is_cuda for t in d)
    for x, y, z in zip(a, b, d):
        assert x.tobytes() == y.tobytes() == z.cpu().numpy().tobytes()
    c1 = m.remove_small_components(dev, min_triangles=10, return_device=True)
    c2 = m.remove_small_components(mesh, min_triangles=10)
    assert all(t.is_cuda for t in c1)
    for x, y in zip(c1, c2):
        assert x.cpu().numpy().tobytes() == y.tobytes()


def test_depth_to_mesh_and_stage(m, tmp_path):
    img, dep = cases.make_image(90, 140, 2), cases.make_depth(97, 151, 2, "scene")
    for refine in (False, True):
        want = CO.remove_small_components(oracle_chain(img, dep, "medium", refine=refine, max_edge=0.3),
                                          min_triangles=10)
        got = m.depth_to_mesh(img, dep, "medium", refine=refine, max_edge=0.3, min_component_triangles=10)
        assert_same(got, want, f"depth_to_mesh {refine}")
    img, dep = cases.make_image(80, 120, 4), cases.make_depth(80, 120, 4, "scene")
    base = m.point_cloud_stage(img, dep, density="high", mesh=True, mesh_preview_voxel=0.05)
    off = m.point_cloud_stage(img, dep, density="high", mesh=True, mesh_preview_voxel=0.05, mesh_min_triangles=None)
    assert base.keys() == off.keys()
    for k, v in base.items():   # the knob left at None changes nothing
        if isinstance(v, np.ndarray):
            assert v.tobytes() == off[k].tobytes(), k
        else:
            assert v == off[k], k
    out = m.point_cloud_stage(img, dep, density="high", mesh=True, mesh_preview_voxel=0.05, mesh_min_triangles=10)
    full = oracle_chain(img, dep, "high", refine=True)
    clusters, n, _ = CO.cluster_connected_triangles(full)
    want = CO.remove_small_components(full, min_triangles=10)
    assert out["mesh_component_count"] == len(n)
    assert out["mesh_removed_triangle_count"] == len(full.triangles) - len(want.triangles) > 0
    assert out["mesh_vertex_count"] == len(want.vertices) and out["mesh_triangle_count"] == len(want.triangles)
    assert out["mesh_file_bytes"] == MO.mesh_ply_bytes(want)
    pre = m.simplify_mesh(want, 0.05)
    assert out["mesh_preview_file_bytes"] == m.mesh_ply_bytes(pre)
    for k, v in base.items():   # the point-cloud outputs are untouched
        if not k.startswith("mesh"):
            assert (v.tobytes() == out[k].tobytes()) if isinstance(v, np.ndarray) else v == out[k], k
    cwd = os.getcwd()
    try:
        os.chdir(tmp_path)
        f = m.point_cloud_stage(img, dep, density="high", mesh=True, mesh_min_triangles=10, filename="scene",
                                return_arrays=False)
        assert open(f["mesh_filepath"], "rb").read() == out["mesh_file_bytes"]
    finally:
        os.chdir(cwd)
