"""CPU: the mesh-smoothing oracle (row m4) against its per-vertex Open3D restatement, known answers, the oracle's
vertex normals against m1's, the shared per-vertex arithmetic (d2pc_smooth.h) on the host against the oracle, and
the argument checks of the Python and C entry points (nothing is launched)."""
import ctypes as C

import numpy as np
import pytest

import image_to_pointcloud_b200 as m
from oracle import d2pc_mesh_oracle as MO
from oracle import d2pc_simplify_oracle as SO
from oracle import d2pc_smooth_oracle as SMO
from tests import components_cases as CC
from tests.hostsmooth import harness as HS
from tests.test_simplify_cpu import lattice_mesh

RUNS = [(method, n) for method in SMO.METHODS for n in (0, 1, 3)]


def same(a, b, what=""):
    for f, x, y in zip(MO.Mesh._fields, a, b):
        if x is None or y is None:
            assert x is None and y is None, f"{what}: {f}"
            continue
        assert x.dtype == y.dtype and x.shape == y.shape, f"{what}: {f} {x.dtype}{x.shape} != {y.dtype}{y.shape}"
        assert x.tobytes() == y.tobytes(), f"{what}: {f}"


def meshes():
    rng = np.random.default_rng(7)
    out = {name: mesh for name, (mesh, _) in CC.hand_meshes().items()}
    for k in range(6):
        V = int(rng.integers(1, 60))
        out[f"soup {k}"] = CC.soup(rng, V, int(rng.integers(0, 2 * V + 5)), normals=k % 2 == 0)
    lat = lattice_mesh(3, R=9, Cc=11)
    out["shuffled lattice"] = CC.shuffled(lat, rng)
    out["simplified"] = SO.simplify_mesh(lattice_mesh(4, R=11, Cc=13), 0.05)
    out["isolated vertices"] = CC.mesh_of(rng.random((7, 3)), [[0, 1, 2]], normals=True)
    return out


@pytest.mark.parametrize("name", list(meshes()))
def test_oracle_forms_agree(name):
    mesh = meshes()[name]
    for method, n in RUNS:
        for scope in SMO.SCOPES:
            want = SMO.filter_smooth(mesh, method, n, scope=scope)
            same(want, SMO.filter_smooth_loop(mesh, method, n, scope=scope), f"{name} {method} {n} {scope}")
            assert want.triangles.tobytes() == np.asarray(mesh.triangles, np.int32).tobytes()
            assert want.vertex_rows.tobytes() == np.asarray(mesh.vertex_rows, np.int64).tobytes()
    same(SMO.compute_vertex_normals(mesh), SMO.compute_vertex_normals_loop(mesh), f"{name} normals")


def test_other_parameters_and_forms():
    mesh = lattice_mesh(5, R=8, Cc=9)
    for lam, mu in ((0.3, -0.31), (1.0, 0.0), (-0.2, 0.7)):
        a = SMO.filter_smooth_taubin(mesh, 2, lam, mu)
        same(a, SMO.filter_smooth_loop(mesh, "taubin", 2, lam, mu), f"{lam} {mu}")
        same(SMO.filter_smooth_laplacian(mesh, 2, lam), SMO.filter_smooth_loop(mesh, "laplacian", 2, lam))
    same(SMO.filter_smooth_simple(mesh, 2), SMO.filter_smooth_loop(mesh, "simple", 2))


def test_adjacency_is_open3d_sets_in_order():
    t = np.array([[0, 0, 1], [2, 3, 4], [4, 3, 2], [1, 5, 5], [6, 6, 6]])
    off, nbr = SMO.adjacency(8, t)
    got = [nbr[off[i]:off[i + 1]].tolist() for i in range(8)]
    assert got == SMO.adjacency_loop(8, t)
    assert got == [[0, 1], [0, 5], [3, 4], [2, 4], [2, 3], [1, 5], [6], []]


def test_known_answers():
    # a planar lattice stays planar under every filter
    x, y = np.meshgrid(np.linspace(-1, 1, 12), np.linspace(-1, 1, 9))
    xyz = np.stack([x.ravel(), y.ravel() ** 3, np.full(x.size, 2.0)], 1).astype(np.float32)
    plane = MO.grid_mesh(xyz, np.zeros_like(xyz), (9, 12), max_angle=90.0)
    assert len(plane.triangles) > 100
    for method in SMO.METHODS:
        out = SMO.filter_smooth(plane, method, 4)
        assert np.abs(out.vertices[:, 2] - 2.0).max() <= 1e-6, method
        assert not np.array_equal(out.vertices, plane.vertices)
    # simple on one triangle: every vertex moves to the centroid
    tri = CC.mesh_of([[0, 0, 0], [3, 0, 0], [0, 6, 3]], [[0, 1, 2]])
    out = SMO.filter_smooth_simple(tri, 1)
    assert np.allclose(out.vertices, [[1, 2, 1]] * 3, rtol=0, atol=1e-6)
    # isolated vertices keep everything, under every method
    mesh = meshes()["isolated vertices"]
    for method, n in RUNS:
        out = SMO.filter_smooth(mesh, method, n)
        assert out.vertices[3:].tobytes() == mesh.vertices[3:].tobytes()
        assert out.colors[3:].tobytes() == mesh.colors[3:].tobytes()
        assert out.vertex_normals[3:].tobytes() == mesh.vertex_normals[3:].tobytes()
    # fields outside the scope are copied; 0 iterations copy everything
    lat = lattice_mesh(2)
    for scope, kept in (("vertex", (1, 3)), ("color", (0, 3)), ("normal", (0, 1))):
        out = SMO.filter_smooth_taubin(lat, 2, scope=scope)
        for f in kept:
            assert out[f].tobytes() == lat[f].tobytes(), (scope, f)
    same(SMO.filter_smooth_taubin(lat, 0), lat, "0 iterations")


def test_vertex_normals_are_grid_mesh_normals():
    for seed in range(4):
        mesh = lattice_mesh(seed, R=10 + seed, Cc=14)
        got = SMO.compute_vertex_normals(mesh._replace(vertex_normals=None))
        assert got.vertex_normals.tobytes() == mesh.vertex_normals.tobytes()
        assert HS.normals(mesh).tobytes() == mesh.vertex_normals.tobytes()
    from tests.test_mesh_cpu import lattice
    z = np.random.default_rng(1).random((20, 30)) + 2
    xyz, rgb = lattice(z, seed=1)
    full = MO.grid_mesh(xyz, rgb, z.shape, max_angle=90.0, remove_unreferenced=False)
    assert SMO.compute_vertex_normals(full).vertex_normals.tobytes() == full.vertex_normals.tobytes()


def test_host_harness_equals_oracle():
    for name, mesh in meshes().items():
        for method, n in RUNS + [("taubin", 10)]:
            for scope in SMO.SCOPES:
                same(HS.smooth(mesh, method, n, scope=scope), SMO.filter_smooth(mesh, method, n, scope=scope),
                     f"{name} {method} {n} {scope}")
        assert HS.normals(mesh).tobytes() == SMO.compute_vertex_normals(mesh).vertex_normals.tobytes(), name


def test_oracle_errors():
    mesh = lattice_mesh(1)
    for bad in ([[0, 1, len(mesh.vertices)]], [[-1, 0, 1]]):
        t = np.concatenate([mesh.triangles, np.asarray(bad, np.int32)])
        with pytest.raises(ValueError, match="vertex that does not exist"):
            SMO.filter_smooth_simple(mesh._replace(triangles=t))
        with pytest.raises(ValueError, match="vertex that does not exist"):
            SMO.compute_vertex_normals(mesh._replace(triangles=t))
    v = mesh.vertices.copy()
    v[4, 2] = np.inf
    with pytest.raises(ValueError, match="non-finite"):
        SMO.filter_smooth_laplacian(mesh._replace(vertices=v))
    c = mesh.colors.copy()
    c[2, 0] = np.nan
    with pytest.raises(ValueError, match="non-finite"):
        SMO.filter_smooth_laplacian(mesh._replace(colors=c))
    SMO.filter_smooth_laplacian(mesh._replace(colors=c), scope="vertex")   # outside the scope: copied
    for kw in (dict(scope="colour"), dict(number_of_iterations=-1), dict(number_of_iterations=1.5),
               dict(lambda_filter=float("nan")), dict(mu=float("inf"))):
        with pytest.raises(ValueError):
            SMO.filter_smooth(mesh, "taubin", **kw)


def test_python_argument_errors():
    mesh = lattice_mesh(6)
    for fn, kw in ((m.filter_smooth_simple, dict(scope="points")), (m.filter_smooth_simple, dict(number_of_iterations=-1)),
                   (m.filter_smooth_laplacian, dict(number_of_iterations=2.5)),
                   (m.filter_smooth_laplacian, dict(lambda_filter=float("nan"))),
                   (m.filter_smooth_taubin, dict(mu=float("-inf")))):
        with pytest.raises(ValueError):
            fn(mesh, **kw)
    img, dep = np.zeros((8, 8, 3), np.uint8), np.ones((8, 8), np.float32)
    with pytest.raises(ValueError, match="mesh=True"):
        m.point_cloud_stage(img, dep, mesh_smooth_iterations=3)
    for bad in (-1, 1.5):
        with pytest.raises(ValueError):
            m.point_cloud_stage(img, dep, mesh=True, mesh_smooth_iterations=bad)


def test_smooth_abi_argument_errors():
    lib = m.load_library()
    nb = C.c_size_t(0)
    V4k, T4k = 3840 * 2160, 2 * 2159 * 3839
    assert lib.d2pc_mesh_smooth_scratch_bytes(V4k, T4k, C.byref(nb)) == 0 and nb.value % 256 == 0
    assert nb.value < 144 * V4k + 100 * T4k   # two float64 states, the edge table, the adjacency
    assert lib.d2pc_mesh_vertex_normals_scratch_bytes(V4k, T4k, C.byref(nb)) == 0 and nb.value < 12 * V4k + 64 * T4k
    for fn in (lib.d2pc_mesh_smooth_scratch_bytes, lib.d2pc_mesh_vertex_normals_scratch_bytes):
        assert fn(0, 0, C.byref(nb)) == 0
        assert fn(2 ** 31, 2 ** 25, C.byref(nb)) == 0
        assert fn(4, (1 << 25) + 1, C.byref(nb)) == 4
        assert fn((1 << 31) + 1, 4, C.byref(nb)) == 4
        assert fn(4, 4, None) == 1
    fake = 1 << 20   # never dereferenced: every call below fails its argument checks first
    ok = dict(xyz=fake, rgb=fake, nrm=fake, V=4, tri=fake, T=4, method=2, iters=3, lam=0.5, mu=-0.53, scope=7,
              scratch=fake, sb=1 << 30, ox=fake, oc=fake, on=fake, err=fake, stream=None)

    def call(**kw):
        return lib.d2pc_mesh_smooth_enqueue(*dict(ok, **kw).values())
    for bad in (dict(method=3), dict(method=-1), dict(scope=0), dict(scope=8), dict(lam=float("nan")),
                dict(mu=float("inf")), dict(xyz=None), dict(rgb=None), dict(tri=None), dict(scratch=None),
                dict(ox=None), dict(oc=None), dict(on=None), dict(nrm=None), dict(err=None), dict(scratch=fake + 16)):
        assert call(**bad) == 1, bad
    assert call(T=(1 << 25) + 1) == 4 and call(V=(1 << 31) + 1) == 4
    assert call(sb=16) == 2
    nok = dict(xyz=fake, V=4, tri=fake, T=4, scratch=fake, sb=1 << 30, on=fake, err=fake, stream=None)

    def ncall(**kw):
        return lib.d2pc_mesh_vertex_normals_enqueue(*dict(nok, **kw).values())
    for bad in (dict(xyz=None), dict(tri=None), dict(scratch=None), dict(on=None), dict(err=None),
                dict(scratch=fake + 16)):
        assert ncall(**bad) == 1, bad
    assert ncall(T=(1 << 25) + 1) == 4
    assert ncall(sb=16) == 2
