"""CPU: the mesh-simplification oracle (row m2) against its per-cluster loop restatement, known answers, and the
argument checks of the Python and C entry points (nothing is launched)."""
import ctypes as C

import numpy as np
import pytest

import image_to_pointcloud_b200 as m
from image_to_pointcloud_b200 import _lib
from oracle import d2pc_mesh_oracle as MO
from oracle import d2pc_simplify_oracle as SO
from tests.simplify_cases import soup
from tests.test_mesh_cpu import assert_mesh_equal, lattice


def lattice_mesh(seed, R=13, Cc=17, normals=True):
    rng = np.random.default_rng(seed)
    z = rng.random((R, Cc)) * 0.5 + 2
    z[rng.random((R, Cc)) < 0.1] += 3
    xyz, rgb = lattice(z, seed=seed)
    return MO.grid_mesh(xyz, rgb, (R, Cc), keep=rng.random(R * Cc) < 0.9, max_angle=89.0, compute_normals=normals)


def both(mesh, vs, contraction):
    a = SO.simplify_mesh(mesh, vs, contraction)
    b = SO.simplify_mesh_loop(mesh, vs, contraction)
    assert_mesh_equal(a, b, f"{vs} {contraction}")
    return a


@pytest.mark.parametrize("contraction", SO.CONTRACTIONS)
def test_vectorised_oracle_equals_loop_on_soups(contraction):
    rng = np.random.default_rng(1 if contraction == "average" else 2)
    for it in range(12):
        mesh = soup(rng, int(rng.integers(1, 60)), int(rng.integers(0, 90)), normals=bool(it % 2), integral=bool(it % 3))
        ext = float(np.ptp(mesh.vertices.astype(np.float64), axis=0).max()) or 1.0
        for f in (1e-3, 0.05, 0.3, 2.0):
            both(mesh, ext * f, contraction)


@pytest.mark.parametrize("contraction", SO.CONTRACTIONS)
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_vectorised_oracle_equals_loop_on_lattices(contraction, seed):
    mesh = lattice_mesh(seed, normals=seed != 1)
    for vs in (0.004, 0.02, 0.05, 0.2):
        out = both(mesh, vs, contraction)
        assert len(out.vertices) <= len(mesh.vertices)


def test_voxel_below_the_spacing_leaves_the_mesh_unchanged():
    mesh = lattice_mesh(4, normals=False)
    out = both(mesh, 1e-5, "average")
    assert_mesh_equal(out, mesh, "unchanged")


def test_voxel_covering_the_mesh_gives_one_vertex():
    mesh = lattice_mesh(5)
    for c in SO.CONTRACTIONS:
        out = both(mesh, 100.0, c)
        assert len(out.vertices) == 1 and len(out.triangles) == 0
        assert out.vertex_rows[0] == mesh.vertex_rows[0]
        assert c == "quadric" or np.allclose(out.vertices[0], mesh.vertices.astype(np.float64).mean(axis=0), atol=1e-6)


def cube_corner(corner=(1.25, -0.5, 2.0), n=4):
    """The three faces of a cube at ``corner`` (x, y, z = corner planes), each an n x n grid of 1/n squares."""
    verts, tris = [], []
    for axis in range(3):
        u, v = [a for a in range(3) if a != axis]
        base = len(verts)
        for i in range(n + 1):
            for j in range(n + 1):
                p = [0.0, 0.0, 0.0]
                p[u], p[v] = i / n, j / n
                verts.append(p)
        for i in range(n):
            for j in range(n):
                a, b, c, d = (base + i * (n + 1) + j, base + (i + 1) * (n + 1) + j, base + i * (n + 1) + j + 1,
                              base + (i + 1) * (n + 1) + j + 1)
                tris += [[a, b, d], [a, d, c]]
    xyz = (np.array(verts) + np.array(corner)).astype(np.float32)
    V = len(xyz)
    return MO.Mesh(xyz, np.full((V, 3), 100.0, np.float32), np.array(tris, np.int32), None, np.arange(V, dtype=np.int64))


def test_quadric_puts_the_cube_corner_on_the_corner():
    mesh = cube_corner()
    d = SO.Detail()
    out = SO.simplify_mesh(mesh, 0.6, "quadric", detail=d)
    assert_mesh_equal(out, SO.simplify_mesh_loop(mesh, 0.6, "quadric"))
    assert d["quadric"][0]
    assert np.abs(d["x"][0] - np.array([1.25, -0.5, 2.0])).max() <= 1e-12
    assert np.array_equal(out.vertices[0], np.array([1.25, -0.5, 2.0], np.float32))
    avg = SO.simplify_mesh(mesh, 0.6, "average")
    assert (avg.vertices[0] > np.array([1.25, -0.5, 2.0], np.float32)).all()   # the mean lies inside the cube


def test_quadric_on_a_plane_falls_back_to_the_average():
    rng = np.random.default_rng(7)
    xy = rng.random((200, 2)) * 2
    xyz = np.concatenate([xy, np.full((200, 1), 0.75)], axis=1).astype(np.float32)
    from scipy.spatial import Delaunay
    tri = Delaunay(xy).simplices.astype(np.int32)
    mesh = MO.Mesh(xyz, np.zeros((200, 3), np.float32), tri, None, np.arange(200, dtype=np.int64))
    d = SO.Detail()
    out = SO.simplify_mesh(mesh, 0.4, "quadric", detail=d)
    assert not d["quadric"].any()
    assert_mesh_equal(out, SO.simplify_mesh(mesh, 0.4, "average"))
    assert (out.vertices[:, 2] == np.float32(0.75)).all()


def test_triangle_with_two_corners_in_one_cluster_counts_twice():
    xyz = np.array([[0.0, 0.0, 1.0], [0.1, 0.0, 1.0], [0.0, 1.0, 0.5]], np.float32)
    mesh = MO.Mesh(xyz, np.zeros((3, 3), np.float32), np.array([[0, 1, 2]], np.int32), None, np.arange(3))
    d = SO.Detail()
    out = SO.simplify_mesh(mesh, 0.5, "quadric", detail=d)
    assert len(out.vertices) == 2 and len(out.triangles) == 0
    q = xyz.astype(np.float64) - xyz.astype(np.float64).min(axis=0)
    c = np.cross(q[1] - q[0], q[2] - q[0])
    area, n = np.linalg.norm(c) / 2, c / np.linalg.norm(c)
    A, b = area * np.outer(n, n), area * -(n @ q[0]) * n
    iu = np.triu_indices(3)
    assert np.allclose(d["A"][0], 2 * A[iu], rtol=1e-14, atol=1e-16)
    assert np.allclose(d["A"][1], A[iu], rtol=1e-14, atol=1e-16)
    assert np.allclose(d["b"][0], 2 * b, rtol=1e-14, atol=1e-16) and np.allclose(d["b"][1], b, rtol=1e-14, atol=1e-16)


def test_rotations_are_merged_and_orientation_twins_kept():
    xyz = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [5, 5, 5]], np.float32)
    tri = np.array([[1, 2, 0], [0, 1, 2], [2, 0, 1], [0, 2, 1], [3, 1, 2], [1, 2, 3]], np.int32)
    mesh = MO.Mesh(xyz, np.zeros((4, 3), np.float32), tri, None, np.arange(4))
    out = both(mesh, 0.01, "average")
    assert out.triangles.tolist() == [[0, 1, 2], [0, 2, 1], [1, 2, 3]]


def test_zero_normal_sum_stays_zero_and_empty_mesh():
    xyz = np.array([[0, 0, 0], [0.01, 0, 0]], np.float32)
    nrm = np.array([[0.0, 0.0, 1.0], [0.0, 0.0, -1.0]])
    mesh = MO.Mesh(xyz, np.zeros((2, 3), np.float32), np.zeros((0, 3), np.int32), nrm, np.arange(2))
    out = both(mesh, 1.0, "average")
    assert np.array_equal(out.vertex_normals, np.zeros((1, 3)))
    empty = MO.Mesh(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int32), None,
                    np.zeros(0, np.int64))
    assert_mesh_equal(both(empty, 0.1, "quadric"), empty)


def test_oracle_errors():
    mesh = lattice_mesh(6)
    for vs in (0.0, -1.0, float("nan"), float("inf")):
        with pytest.raises(ValueError):
            SO.simplify_mesh(mesh, vs)
    with pytest.raises(ValueError):
        SO.simplify_mesh(mesh, 0.1, "median")
    ext = float(np.ptp(mesh.vertices.astype(np.float64), axis=0).max())
    with pytest.raises(ValueError, match="too small"):
        SO.simplify_mesh(mesh, ext / 2 ** 22)
    bad = mesh._replace(triangles=np.concatenate([mesh.triangles, [[0, 1, len(mesh.vertices)]]]).astype(np.int32))
    with pytest.raises(ValueError):
        SO.simplify_mesh(bad, 0.1)
    v = mesh.vertices.copy()
    v[3, 1] = np.nan
    with pytest.raises(ValueError):
        SO.simplify_mesh(mesh._replace(vertices=v), 0.1)


def test_python_argument_errors():
    mesh = lattice_mesh(6)
    for kw in (dict(voxel_size=0.0), dict(voxel_size=float("nan")), dict(voxel_size=-2.0),
               dict(voxel_size=0.1, contraction="median")):
        with pytest.raises(ValueError):
            m.simplify_mesh(mesh, **kw)
    with pytest.raises(ValueError, match="mesh=True"):
        m.point_cloud_stage(np.zeros((8, 8, 3), np.uint8), np.ones((8, 8), np.float32), mesh_preview_voxel=0.1)
    with pytest.raises(ValueError):
        m.point_cloud_stage(np.zeros((8, 8, 3), np.uint8), np.ones((8, 8), np.float32), mesh=True,
                            mesh_preview_voxel=0.0)
    assert _lib.SIMPLIFY_QUADRIC == 1 and _lib.SIMPLIFY_NORMALS == 2


def test_simplify_abi_argument_errors():
    lib = m.load_library()
    nb = C.c_size_t(0)
    assert lib.d2pc_mesh_simplify_scratch_bytes(1_750_000, 2_120_000, C.byref(nb)) == 0 and nb.value % 256 == 0
    assert lib.d2pc_mesh_simplify_scratch_bytes(0, 0, C.byref(nb)) == 0
    assert lib.d2pc_mesh_simplify_scratch_bytes(1 << 24, 0, C.byref(nb)) == 4
    assert lib.d2pc_mesh_simplify_scratch_bytes(4, 1 << 31, C.byref(nb)) == 4
    assert lib.d2pc_mesh_simplify_scratch_bytes(4, 4, None) == 1
    fake = 1 << 20   # never dereferenced: every call below fails its argument checks first
    ok = dict(xyz=fake, rgb=fake, nrm=fake, row=fake, V=4, tri=fake, T=4, vs=0.1, flags=3, scratch=fake, sb=1 << 30,
              ox=fake, oc=fake, on=fake, orow=fake, vcnt=fake, otri=fake, tcnt=fake, err=fake, stream=None)

    def call(**kw):
        a = dict(ok, **kw)
        return lib.d2pc_mesh_simplify_enqueue(*a.values())
    for bad in (dict(vs=0.0), dict(vs=float("nan")), dict(vs=float("inf")), dict(flags=4), dict(xyz=None),
                dict(rgb=None), dict(row=None), dict(nrm=None), dict(on=None), dict(tri=None), dict(otri=None),
                dict(scratch=None), dict(vcnt=None), dict(tcnt=None), dict(err=None), dict(ox=None),
                dict(scratch=fake + 16)):
        assert call(**bad) == 1, bad
    assert call(V=1 << 24) == 4 and call(T=1 << 31) == 4
    assert call(sb=16) == 2
