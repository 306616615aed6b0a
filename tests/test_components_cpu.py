"""CPU: the mesh-components oracle (row m3) against its BFS restatement, the fixed-point areas against math.fsum,
the shared union-find steps (d2pc_components.h) on the host in random orders, and the argument checks of the Python
and C entry points (nothing is launched)."""
import ctypes as C
import math

import numpy as np
import pytest

import image_to_pointcloud_b200 as m
from oracle import d2pc_components_oracle as CO
from oracle import d2pc_mesh_oracle as MO
from tests import components_cases as CC
from tests.hostcomp import harness as HC
from tests.test_simplify_cpu import lattice_mesh


def both(mesh, what="", seed=None):
    a = CO.cluster_connected_triangles(mesh)
    b = CO.cluster_connected_triangles_loop(mesh, None if seed is None else np.random.default_rng(seed))
    for x, y, name in zip(a, b, ("clusters", "n", "area")):
        assert x.dtype == y.dtype and x.tobytes() == y.tobytes(), f"{what}: {name}"
    CC.check_areas(mesh, *a)
    return a


def lattice_meshes():
    out = [lattice_mesh(s, R=13 + s, Cc=17 + 2 * s, normals=s % 2 == 0) for s in range(4)]
    rng = np.random.default_rng(5)
    z = rng.random((30, 40)) * 0.3 + 2
    z[rng.random(z.shape) < 0.3] += 4   # many islands
    from tests.test_mesh_cpu import lattice
    xyz, rgb = lattice(z, seed=5)
    out.append(MO.grid_mesh(xyz, rgb, z.shape, max_angle=60.0))
    return out


@pytest.mark.parametrize("name", list(CC.hand_meshes()))
def test_hand_meshes(name):
    mesh, want = CC.hand_meshes()[name]
    clusters, n, area = both(mesh, name, seed=1)
    assert clusters.tolist() == want
    assert n.tolist() == np.bincount(np.asarray(want, np.int64), minlength=len(n)).tolist()
    for seed in range(5):
        lab, hn, ha, err = HC.components(mesh, seed)
        assert err == 0 and lab.tobytes() == clusters.tobytes() and hn.tobytes() == n.tobytes()
        assert ha.tobytes() == area.tobytes()


def test_oracle_forms_agree_on_soups_and_lattices():
    rng = np.random.default_rng(2)
    for it in range(40):
        V = int(rng.integers(1, 80))
        mesh = CC.soup(rng, V, int(rng.integers(0, 2 * V + 5)))
        both(mesh, f"soup {it}", seed=it)
    for k, mesh in enumerate(lattice_meshes()):
        clusters, n, _ = both(mesh, f"lattice {k}", seed=k)
        assert (np.diff(np.unique(clusters, return_index=True)[1]) > 0).all()   # numbered by lowest triangle
        assert n.sum() == len(mesh.triangles)


def test_numbering_follows_the_lowest_triangle_under_shuffles():
    rng = np.random.default_rng(3)
    mesh = lattice_meshes()[-1]
    clusters, n, _ = both(mesh)
    assert len(n) > 5
    for it in range(3):
        sh = CC.shuffled(mesh, rng)
        c2, n2, _ = both(sh, f"shuffle {it}")
        assert sorted(n2.tolist()) == sorted(n.tolist())
        first = np.unique(c2, return_index=True)[1]
        assert (np.diff(first) > 0).all()


def test_fixed_point_area_rule():
    mesh = CC.mesh_of([[0, 0, 0], [3, 0, 0], [0, 4, 0], [1e-3, 0, 0], [0, 1e-3, 0]], [[0, 1, 2], [0, 3, 4]])
    clusters, n, area = both(mesh)
    assert clusters.tolist() == [0, 1] and area[0] == 6.0
    a = CO.triangle_areas(mesh.vertices, mesh.triangles.astype(np.int64))
    assert math.frexp(6.0)[1] == 3
    assert CO.area_scale(a) == 2.0 ** (62 - 3 - 1)
    assert area[1] == float(int(np.rint(a[1] * 2.0 ** 58))) / 2.0 ** 58
    zero = CC.mesh_of([[1, 1, 1]] * 3, [[0, 1, 2], [0, 1, 2]])
    z = both(zero)
    assert z[2].tolist() == [0.0] and CO.area_scale(np.zeros(2)) == 2.0 ** 61


def test_errors():
    mesh = lattice_mesh(1)
    for bad in ([[0, 1, len(mesh.vertices)]], [[-1, 0, 1]]):
        t = np.concatenate([mesh.triangles, np.asarray(bad, np.int32)])
        with pytest.raises(ValueError, match="vertex that does not exist"):
            CO.cluster_connected_triangles(mesh._replace(triangles=t))
        lab, n, area, err = HC.components(mesh._replace(triangles=t), 0)
        assert err == 1 and len(n) == 0
    v = mesh.vertices.copy()
    v[4, 2] = np.inf
    with pytest.raises(ValueError, match="non-finite"):
        CO.cluster_connected_triangles(mesh._replace(vertices=v))
    assert HC.components(mesh._replace(vertices=v), 0)[3] == 2
    empty = CC.mesh_of(np.zeros((0, 3)), [[0, 0, 0]])
    with pytest.raises(ValueError):
        CO.cluster_connected_triangles(empty)
    assert HC.components(empty, 0)[3] == 1


def test_host_harness_random_orders():
    rng = np.random.default_rng(4)
    meshes = lattice_meshes() + [CC.strip(301), CC.comb(12, 9), CC.edge_fan(500), CC.isolated(300)]
    meshes += [CC.soup(rng, int(rng.integers(2, 200)), int(rng.integers(1, 500))) for _ in range(20)]
    for k, mesh in enumerate(meshes):
        want = CO.cluster_connected_triangles(mesh)
        for seed in range(4):
            lab, n, area, err = HC.components(mesh, 1000 * k + seed)
            assert err == 0, (k, seed, err)
            assert lab.tobytes() == want[0].tobytes() and n.tobytes() == want[1].tobytes(), (k, seed)
            assert area.tobytes() == want[2].tobytes(), (k, seed)


def test_host_harness_bounds():
    lib = HC.load()
    assert lib.hc_insert_full(1024) == 1   # a full table returns the failure instead of probing forever
    assert lib.hc_chain_bounds(1000) == 1  # find and unite stop at their bound


def test_removal_oracle():
    rng = np.random.default_rng(6)
    mesh = lattice_mesh(2)
    T = len(mesh.triangles)
    for mask in (np.zeros(T, bool), np.ones(T, bool), rng.random(T) < 0.5):
        out = CO.remove_triangles_by_mask(mesh, mask)
        assert np.array_equal(out.triangles.shape, ((~mask).sum(), 3))
        used = np.unique(mesh.triangles[~mask])
        assert np.array_equal(out.vertex_rows, mesh.vertex_rows[used])
        assert np.array_equal(out.vertices[out.triangles], mesh.vertices[mesh.triangles[~mask]])
        keep_all = CO.remove_triangles_by_mask(mesh, mask, remove_unreferenced=False)
        assert np.array_equal(keep_all.triangles, mesh.triangles[~mask])
        assert keep_all.vertex_normals.tobytes() == mesh.vertex_normals.tobytes()
    small = lattice_meshes()[-1]
    clusters, n, _ = CO.cluster_connected_triangles(small)
    out = CO.remove_small_components(small, min_triangles=10)
    assert len(out.triangles) == int(n[n >= 10].sum())
    assert len(CO.cluster_connected_triangles(out)[1]) == int((n >= 10).sum())


def test_python_argument_errors():
    mesh = lattice_mesh(6)
    for kw in (dict(), dict(min_triangles=0), dict(min_triangles=2.5), dict(min_area=float("nan"))):
        with pytest.raises(ValueError):
            m.remove_small_components(mesh, **kw)
    img, dep = np.zeros((8, 8, 3), np.uint8), np.ones((8, 8), np.float32)
    with pytest.raises(ValueError, match="mesh=True"):
        m.point_cloud_stage(img, dep, mesh_min_triangles=10)
    for bad in (0, -3):
        with pytest.raises(ValueError):
            m.point_cloud_stage(img, dep, mesh=True, mesh_min_triangles=bad)
        with pytest.raises(ValueError):
            m.depth_to_mesh(img, dep, min_component_triangles=bad)


def test_components_abi_argument_errors():
    lib = m.load_library()
    nb = C.c_size_t(0)
    T4k = 2 * 2159 * 3839
    assert lib.d2pc_mesh_components_scratch_bytes(8_300_000, T4k, C.byref(nb)) == 0 and nb.value % 256 == 0
    assert nb.value < 96 * T4k   # 84 bytes a triangle
    assert lib.d2pc_mesh_components_scratch_bytes(0, 0, C.byref(nb)) == 0
    assert lib.d2pc_mesh_components_scratch_bytes(4, (1 << 25) + 1, C.byref(nb)) == 4
    assert lib.d2pc_mesh_components_scratch_bytes((1 << 31) + 1, 4, C.byref(nb)) == 4
    assert lib.d2pc_mesh_components_scratch_bytes(4, 4, None) == 1
    assert lib.d2pc_mesh_filter_scratch_bytes(8_300_000, T4k, C.byref(nb)) == 0 and nb.value % 256 == 0
    assert lib.d2pc_mesh_filter_scratch_bytes(4, (1 << 25) + 1, C.byref(nb)) == 4
    assert lib.d2pc_mesh_filter_scratch_bytes(4, 4, None) == 1
    fake = 1 << 20   # never dereferenced: every call below fails its argument checks first
    ok = dict(xyz=fake, V=4, tri=fake, T=4, scratch=fake, sb=1 << 30, lab=fake, n=fake, area=fake, k=fake, err=fake,
              stream=None)

    def call(**kw):
        return lib.d2pc_mesh_components_enqueue(*dict(ok, **kw).values())
    for bad in (dict(xyz=None), dict(tri=None), dict(scratch=None), dict(lab=None), dict(n=None), dict(area=None),
                dict(k=None), dict(err=None), dict(scratch=fake + 16)):
        assert call(**bad) == 1, bad
    assert call(T=(1 << 25) + 1) == 4 and call(V=(1 << 31) + 1) == 4
    assert call(sb=16) == 2
    fok = dict(xyz=fake, rgb=fake, nrm=fake, row=fake, V=4, tri=fake, T=4, keep=fake, flags=3, scratch=fake,
               sb=1 << 30, ox=fake, oc=fake, on=fake, orow=fake, vcnt=fake, otri=fake, tcnt=fake, err=fake,
               stream=None)

    def fcall(**kw):
        return lib.d2pc_mesh_filter_enqueue(*dict(fok, **kw).values())
    for bad in (dict(flags=4), dict(xyz=None), dict(rgb=None), dict(row=None), dict(nrm=None), dict(on=None),
                dict(tri=None), dict(keep=None), dict(otri=None), dict(scratch=None), dict(vcnt=None),
                dict(tcnt=None), dict(err=None), dict(ox=None), dict(scratch=fake + 16)):
        assert fcall(**bad) == 1, bad
    assert fcall(T=(1 << 25) + 1) == 4
    assert fcall(sb=16) == 2
