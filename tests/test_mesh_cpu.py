"""CPU: the lattice-mesh oracle (row m1) against its per-quad loop restatement, its geometric properties, the mesh PLY
layout, and the host-side argument checks of the mesh entry points (nothing is launched)."""
import ctypes as C

import numpy as np
import pytest

import image_to_pointcloud_b200 as m
from image_to_pointcloud_b200 import _lib
from oracle import d2pc_mesh_oracle as MO
from oracle.d2pc_normals_oracle import PLY_NORMAL_RECORD_DTYPE
from oracle.d2pc_oracle import PLY_RECORD_DTYPE


def lattice(z, f=100.0, seed=0):
    """Emit-like rows of an R x C depth lattice z (float64): x = (u - cx) z / f, y = (v - cy) z / f."""
    R, Cc = z.shape
    v, u = np.mgrid[0:R, 0:Cc].astype(np.float64)
    xyz = np.stack([(u - Cc / 2) * z / f, (v - R / 2) * z / f, z], -1).reshape(-1, 3).astype(np.float32)
    rgb = np.random.default_rng(seed).integers(0, 256, (R * Cc, 3)).astype(np.float32)
    return xyz, rgb


def assert_mesh_equal(a, b, what=""):
    for f in MO.Mesh._fields:
        x, y = getattr(a, f), getattr(b, f)
        if x is None or y is None:
            assert x is None and y is None, f"{what}: {f}"
            continue
        assert x.shape == y.shape and x.dtype == y.dtype, f"{what}: {f} {x.shape}/{x.dtype} != {y.shape}/{y.dtype}"
        assert x.tobytes() == y.tobytes(), f"{what}: {f} differs"


def random_case(rng, R, Cc):
    z = rng.random((R, Cc)) * 3 + 1
    if rng.random() < 0.6:                                   # depth steps
        z[rng.random((R, Cc)) < 0.2] += 6
    xyz, rgb = lattice(z, seed=int(rng.integers(1 << 30)))
    xyz[rng.random(R * Cc) < 0.08] = np.nan                  # NaN rows
    xyz[rng.random(R * Cc) < 0.02, 1] = np.inf
    keep = rng.random(R * Cc) < 0.9 if rng.random() < 0.5 else None   # holes
    return xyz, rgb, keep


@pytest.mark.parametrize("shape", [(1, 1), (1, 9), (9, 1), (2, 2), (3, 4), (7, 5), (12, 17)])
def test_vectorised_oracle_equals_loop(shape):
    rng = np.random.default_rng(shape[0] * 100 + shape[1])
    for it in range(24):
        xyz, rgb, keep = random_case(rng, *shape)
        kw = dict(keep=keep, max_edge=(None, 0.4, 3.0)[it % 3], max_angle=(85.0, 90.0, 60.0, 30.0)[it % 4],
                  remove_unreferenced=bool(it % 2), compute_normals=bool(it % 5))
        assert_mesh_equal(MO.grid_mesh(xyz, rgb, shape, **kw), MO.grid_mesh_loop(xyz, rgb, shape, **kw), f"{shape} {it}")


def test_all_dropped_lattice():
    xyz, rgb = lattice(np.full((4, 5), 2.0))
    for keep in (np.zeros(20, bool), None):
        p = xyz.copy() if keep is not None else np.full_like(xyz, np.nan)
        for ru in (True, False):
            a = MO.grid_mesh(p, rgb, (4, 5), keep=keep, remove_unreferenced=ru)
            assert_mesh_equal(a, MO.grid_mesh_loop(p, rgb, (4, 5), keep=keep, remove_unreferenced=ru))
            assert a.vertices.shape == (0, 3) and a.triangles.shape == (0, 3) and a.vertex_normals.shape == (0, 3)


def test_fronto_parallel_plane_is_complete_and_faces_the_camera():
    R, Cc = 6, 9
    xyz, rgb = lattice(np.full((R, Cc), 2.5))
    mesh = MO.grid_mesh(xyz, rgb, (R, Cc))
    assert len(mesh.triangles) == 2 * (R - 1) * (Cc - 1)
    assert len(mesh.vertices) == R * Cc and np.array_equal(mesh.vertex_rows, np.arange(R * Cc))
    assert (mesh.vertex_normals == np.array([0.0, 0.0, -1.0])).all()


def test_depth_step_removed_at_85_and_kept_at_90():
    z = np.full((6, 10), 2.0)
    z[:, 5:] = 8.0                                           # a wall-to-background step between columns 4 and 5
    xyz, rgb = lattice(z)
    full = 2 * 5 * 9
    at85 = MO.grid_mesh(xyz, rgb, (6, 10), max_angle=85.0)
    at90 = MO.grid_mesh(xyz, rgb, (6, 10), max_angle=90.0)
    assert len(at90.triangles) == full
    assert len(at85.triangles) == full - 2 * 5               # the quads across the step are gone
    rows = at85.vertex_rows[at85.triangles]                  # no kept triangle spans the step
    cols = rows % 10
    assert not ((cols.min(axis=1) <= 4) & (cols.max(axis=1) >= 5)).any()


def test_edges_are_consistently_oriented():
    rng = np.random.default_rng(5)
    for _ in range(10):
        xyz, rgb, keep = random_case(rng, 11, 13)
        t = MO.grid_mesh(xyz, rgb, (11, 13), keep=keep, max_angle=89.0).triangles.astype(np.int64)
        directed = np.concatenate([t[:, [0, 1]], t[:, [1, 2]], t[:, [2, 0]]])
        _, cnt = np.unique(directed, axis=0, return_counts=True)
        assert cnt.max(initial=0) <= 1
        _, cnt = np.unique(np.sort(directed, axis=1), axis=0, return_counts=True)
        assert cnt.max(initial=0) <= 2


@pytest.mark.parametrize("normals", [True, False])
def test_mesh_ply_parses_back(normals):
    rng = np.random.default_rng(3)
    xyz, rgb, keep = random_case(rng, 9, 8)
    mesh = MO.grid_mesh(xyz, rgb, (9, 8), keep=keep, compute_normals=normals)
    data = MO.mesh_ply_bytes(mesh)
    head_end = data.index(b"end_header\n") + len(b"end_header\n")
    head = data[:head_end].decode("ascii")
    nv, nt = len(mesh.vertices), len(mesh.triangles)
    assert f"element vertex {nv}\n" in head and f"element face {nt}\nproperty list uchar uint vertex_indices\n" in head
    assert head == (MO.PLY_MESH_NORMAL_HEADER if normals else MO.PLY_MESH_HEADER).format(n=nv, m=nt)
    assert head == (m.writers.PLY_MESH_NORMAL_HEADER if normals else m.writers.PLY_MESH_HEADER).format(n=nv, m=nt)
    vdt = PLY_NORMAL_RECORD_DTYPE if normals else PLY_RECORD_DTYPE
    body = data[head_end:]
    assert len(body) == nv * vdt.itemsize + nt * 13
    v = np.frombuffer(body[:nv * vdt.itemsize], vdt)
    f = np.frombuffer(body[nv * vdt.itemsize:], MO.PLY_FACE_RECORD_DTYPE)
    assert np.array_equal(np.stack([v["x"], v["y"], v["z"]], 1), mesh.vertices.astype(np.float64))
    if normals:
        assert np.array_equal(np.stack([v["nx"], v["ny"], v["nz"]], 1), mesh.vertex_normals)
    assert (f["n"] == 3).all()
    assert np.array_equal(np.stack([f["v0"], f["v1"], f["v2"]], 1).astype(np.int64), mesh.triangles.astype(np.int64))


def test_mesh_abi_argument_errors():
    lib = m.load_library()
    nb = C.c_size_t(0)
    assert lib.d2pc_grid_mesh_scratch_bytes(1080, 1920, C.byref(nb)) == 0 and nb.value > 0 and nb.value % 256 == 0
    assert lib.d2pc_grid_mesh_scratch_bytes(1, 1, C.byref(nb)) == 0
    assert lib.d2pc_grid_mesh_scratch_bytes(0, 5, C.byref(nb)) == 1
    assert lib.d2pc_grid_mesh_scratch_bytes(5, 0, C.byref(nb)) == 1
    assert lib.d2pc_grid_mesh_scratch_bytes(1 << 16, 1 << 15, C.byref(nb)) == 1   # R * C = 2^31
    assert lib.d2pc_grid_mesh_scratch_bytes(4, 4, None) == 1
    fake = 1 << 20   # never dereferenced: every call below fails its argument checks first
    ok = dict(xyz=fake, rgb=fake, keep=None, rows=4, cols=4, max_edge=0.0, cos2=0.0076, flags=3, scratch=fake,
              sb=1 << 20, vx=fake, vc=fake, vr=fake, vn=fake, vcnt=fake, tri=fake, tcnt=fake, stream=None)

    def call(**kw):
        a = dict(ok, **kw)
        return lib.d2pc_grid_mesh_enqueue(*a.values())
    for bad in (dict(xyz=None), dict(rgb=None), dict(scratch=None), dict(vx=None), dict(vcnt=None), dict(tcnt=None),
                dict(rows=0), dict(cols=0), dict(rows=1 << 16, cols=1 << 15), dict(flags=4), dict(vn=None),
                dict(tri=None), dict(cos2=-0.1), dict(cos2=1.5), dict(cos2=float("nan")),
                dict(max_edge=float("nan")), dict(max_edge=float("inf")), dict(scratch=fake + 16)):
        assert call(**bad) == 1, bad
    assert call(sb=16) == 2                                                   # workspace too small
    assert lib.d2pc_ply_face_records_enqueue(None, fake, 4, fake, None) == 1
    assert lib.d2pc_ply_face_records_enqueue(fake, None, 4, fake, None) == 1
    assert lib.d2pc_ply_face_records_enqueue(fake, fake, 0, fake, None) == 1
    assert lib.d2pc_ply_face_records_enqueue(fake, fake, 4, fake + 4, None) == 1   # records not 16-byte aligned


def test_python_argument_errors():
    xyz, rgb = lattice(np.full((3, 3), 1.0))
    for kw in (dict(max_angle=0.0), dict(max_angle=91.0), dict(max_edge=-1.0), dict(max_edge=float("nan"))):
        with pytest.raises(ValueError):
            m.grid_mesh(xyz, rgb, (3, 3), **kw)
    with pytest.raises(ValueError):
        m.grid_mesh(xyz, rgb, (0, 3))
    assert _lib.MESH_REMOVE_UNREFERENCED == 1 and _lib.MESH_NORMALS == 2
