"""GPU (-m gpu): mesh smoothing (filter_smooth_simple / _laplacian / _taubin), compute_vertex_normals and
point_cloud_stage(mesh_smooth_iterations=...) against the oracle (oracle/d2pc_smooth_oracle.py), bit for bit: float32
words of vertices and colours, float64 words of normals, unchanged triangles and vertex rows."""
import os

import numpy as np
import pytest

from oracle import d2pc_components_oracle as CO
from oracle import d2pc_mesh_oracle as MO
from oracle import d2pc_simplify_oracle as SO
from oracle import d2pc_smooth_oracle as SMO
from tests import cases
from tests import components_cases as CC
from tests.test_mesh_gpu import assert_same, oracle_chain, stage_lattice

pytestmark = pytest.mark.gpu

FUNCS = {"simple": "filter_smooth_simple", "laplacian": "filter_smooth_laplacian", "taubin": "filter_smooth_taubin"}


@pytest.fixture(scope="module")
def m():
    import torch
    assert torch.cuda.is_available()
    import image_to_pointcloud_b200 as mod
    mod.load_library()
    return mod


def smooth(m, mesh, method, n, scope="all", **kw):
    return getattr(m, FUNCS[method])(mesh, n, scope=scope, **kw)


def run(m, mesh, method, n, scope="all", what=""):
    want = SMO.filter_smooth(mesh, method, n, scope=scope)
    assert_same(smooth(m, mesh, method, n, scope), want, f"{what} {method} {n} {scope}")
    return want


def run_all(m, mesh, what, iterations=(0, 1, 3, 10)):
    for method in SMO.METHODS:
        for n in iterations:
            for scope in SMO.SCOPES:
                run(m, mesh, method, n, scope, what)
    assert_same(m.compute_vertex_normals(mesh), SMO.compute_vertex_normals(mesh), f"{what} normals")


def star(n):
    """A hub (vertex 0) with n spokes: the hub has n neighbours and n triangles."""
    a = np.linspace(0, 2 * np.pi, n, endpoint=False)
    xyz = np.concatenate([[[0, 0, 0.3]], np.stack([np.cos(a), np.sin(a), 0.1 * np.cos(3 * a)], 1)])
    k = np.arange(n)
    return CC.mesh_of(xyz, np.stack([np.zeros(n, np.int64), k + 1, (k + 1) % n + 1], 1))


@pytest.mark.parametrize("kind", ["uniform", "scene", "ties"])
@pytest.mark.parametrize("density", ["high", "medium"])
def test_stage_lattices(m, kind, density):
    _, _, xyz, rgb, shape = stage_lattice(97, 151, 3, kind, density)
    keep = np.random.default_rng(11).random(len(xyz)) < 0.85
    rng = np.random.default_rng(12)
    for k, mesh in enumerate((MO.grid_mesh(xyz, rgb, shape), MO.grid_mesh(xyz, rgb, shape, keep=keep, max_angle=70.0))):
        run_all(m, mesh, f"{kind} {density} {k}")
        assert m.compute_vertex_normals(mesh).vertex_normals.tobytes() == mesh.vertex_normals.tobytes()
        run_all(m, CC.shuffled(mesh, rng), f"{kind} {density} {k} shuffled", (1, 3))
        run_all(m, SO.simplify_mesh(mesh, 0.02), f"{kind} {density} {k} simplified", (1, 3))


def test_hand_meshes_soups_and_empty(m):
    for name, (mesh, _) in CC.hand_meshes().items():
        run_all(m, mesh, name, (0, 1, 3))
    rng = np.random.default_rng(3)
    for it in range(12):
        V = int(rng.integers(1, 3000))
        run_all(m, CC.soup(rng, V, int(rng.integers(0, 3 * V)), normals=it % 2 == 0), f"soup {it}", (1, 3))
    iso = CC.mesh_of(rng.random((50, 3)), [[0, 1, 2], [2, 3, 4], [2, 2, 5]], normals=True)
    run_all(m, iso, "isolated vertices", (1, 3))
    pts = CC.mesh_of(rng.random((40, 3)), np.zeros((0, 3)), normals=True)
    run_all(m, pts, "no triangles", (0, 2))
    out = m.compute_vertex_normals(pts)
    assert (out.vertex_normals == [0.0, 0.0, 1.0]).all()
    empty = CC.mesh_of(np.zeros((0, 3)), np.zeros((0, 3)))
    for method in SMO.METHODS:
        out = smooth(m, empty, method, 2)
        assert len(out.vertices) == 0 and len(out.triangles) == 0
    assert len(m.compute_vertex_normals(empty).vertex_normals) == 0


def test_large_degrees(m):
    # the hub's segment on every sort path: own thread (<= 32), a CTA in shared memory (<= 4096), global memory
    for n in (32, 33, 4096, 4097):
        mesh = star(n)
        for method in SMO.METHODS:
            run(m, mesh, method, 2, what=f"star {n}")
        assert_same(m.compute_vertex_normals(mesh), SMO.compute_vertex_normals(mesh), f"star {n} normals")
    fan = CC.edge_fan(10_000)
    for method in SMO.METHODS:
        run(m, fan, method, 1, what="fan")
    assert_same(m.compute_vertex_normals(fan), SMO.compute_vertex_normals(fan), "fan normals")
    big = star(1 << 17)
    run(m, big, "simple", 1, what="star 2^17")
    run(m, big, "taubin", 1, what="star 2^17")
    assert_same(m.compute_vertex_normals(big), SMO.compute_vertex_normals(big), "star 2^17 normals")


def test_full_1080p_high_scene_mesh(m):
    img, dep = cases.make_image(1080, 1920, 1), cases.make_depth(1080, 1920, 1, "scene")
    mesh = m.depth_to_mesh(img, dep, "high")
    assert len(mesh.triangles) > 2_000_000
    want = run(m, mesh, "taubin", 10, what="1080p high")
    run(m, mesh, "taubin", 10, "vertex", what="1080p high")
    assert m.compute_vertex_normals(mesh).vertex_normals.tobytes() == mesh.vertex_normals.tobytes()
    nrm = m.compute_vertex_normals(want)
    assert nrm.vertex_normals.tobytes() == SMO.compute_vertex_normals(want).vertex_normals.tobytes()


def test_refused_meshes(m):
    mesh = CC.soup(np.random.default_rng(4), 50, 80, normals=True)
    for bad in ([[0, 1, 50]], [[-1, 1, 2]]):
        t = np.concatenate([mesh.triangles, np.asarray(bad, np.int32)])
        for method in SMO.METHODS:
            with pytest.raises(ValueError, match="vertex that does not exist"):
                smooth(m, mesh._replace(triangles=t), method, 1)
        with pytest.raises(ValueError, match="vertex that does not exist"):
            m.compute_vertex_normals(mesh._replace(triangles=t))
    v = mesh.vertices.copy()
    v[7, 1] = np.nan
    with pytest.raises(ValueError, match="non-finite"):
        m.filter_smooth_taubin(mesh._replace(vertices=v))
    with pytest.raises(ValueError, match="non-finite"):
        m.compute_vertex_normals(mesh._replace(vertices=v))
    nrm = mesh.vertex_normals.copy()
    nrm[3, 0] = np.inf
    with pytest.raises(ValueError, match="non-finite"):
        m.filter_smooth_laplacian(mesh._replace(vertex_normals=nrm))
    run(m, mesh._replace(vertex_normals=nrm), "laplacian", 2, "vertex", "normal outside the scope")
    empty = CC.mesh_of(np.zeros((0, 3)), np.zeros((0, 3)))
    with pytest.raises(ValueError, match="vertex that does not exist"):
        m.filter_smooth_simple(empty._replace(triangles=np.zeros((1, 3), np.int32)))
    for kw in (dict(scope="xyz"), dict(number_of_iterations=-2), dict(lambda_filter=float("nan"))):
        with pytest.raises(ValueError):
            m.filter_smooth_laplacian(mesh, **kw)


def test_device_tensors_and_repeatability(m):
    import torch
    img, dep = cases.make_image(240, 320, 6), cases.make_depth(240, 320, 6, "scene")
    mesh = m.depth_to_mesh(img, dep, "high")
    dev = m.TriangleMesh(*(torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in mesh))
    a, b = m.filter_smooth_taubin(mesh, 5), m.filter_smooth_taubin(mesh, 5)
    d = m.filter_smooth_taubin(dev, 5, return_device=True)
    assert all(t.is_cuda for t in d)
    for x, y, z in zip(a, b, d):
        assert x.tobytes() == y.tobytes() == z.cpu().numpy().tobytes()
    n1 = m.compute_vertex_normals(dev, return_device=True)
    assert all(t.is_cuda for t in n1)
    assert n1.vertex_normals.cpu().numpy().tobytes() == mesh.vertex_normals.tobytes()


def oracle_stage_mesh(img, dep, iterations, min_triangles=None):
    full = oracle_chain(img, dep, "high", refine=True)
    if min_triangles is not None:
        full = CO.remove_small_components(full, min_triangles=min_triangles)
    return SMO.compute_vertex_normals(SMO.filter_smooth_taubin(full, iterations, scope="vertex"))


def test_stage(m, tmp_path):
    img, dep = cases.make_image(80, 120, 4), cases.make_depth(80, 120, 4, "scene")
    base = m.point_cloud_stage(img, dep, density="high", mesh=True, mesh_preview_voxel=0.05, mesh_min_triangles=10)
    off = m.point_cloud_stage(img, dep, density="high", mesh=True, mesh_preview_voxel=0.05, mesh_min_triangles=10,
                              mesh_smooth_iterations=None)
    assert base.keys() == off.keys()
    for k, v in base.items():   # the knob left at None changes nothing
        assert (v.tobytes() == off[k].tobytes()) if isinstance(v, np.ndarray) else v == off[k], k
    for n, kw in ((10, {}), (3, dict(mesh_min_triangles=10)), (10, dict(mesh_min_triangles=10, mesh_preview_voxel=0.05)),
                  (0, {})):
        out = m.point_cloud_stage(img, dep, density="high", mesh=True, mesh_smooth_iterations=n, **kw)
        want = oracle_stage_mesh(img, dep, n, kw.get("mesh_min_triangles"))
        assert out["mesh_vertex_count"] == len(want.vertices) and out["mesh_triangle_count"] == len(want.triangles)
        assert out["mesh_file_bytes"] == MO.mesh_ply_bytes(want), (n, kw)
        if "mesh_preview_voxel" in kw:
            assert out["mesh_preview_file_bytes"] == m.mesh_ply_bytes(m.simplify_mesh(want, 0.05))
        for k, v in base.items():   # the point-cloud outputs are untouched
            if not k.startswith("mesh"):
                assert (v.tobytes() == out[k].tobytes()) if isinstance(v, np.ndarray) else v == out[k], k
    cwd = os.getcwd()
    try:
        os.chdir(tmp_path)
        f = m.point_cloud_stage(img, dep, density="high", mesh=True, mesh_smooth_iterations=10, filename="scene",
                                return_arrays=False)
        assert open(f["mesh_filepath"], "rb").read() == MO.mesh_ply_bytes(oracle_stage_mesh(img, dep, 10))
    finally:
        os.chdir(cwd)
