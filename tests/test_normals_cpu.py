"""CPU: the normals spec (oracle/d2pc_normals_oracle.py, Open3D estimate_normals restated) checked against known
answers, the 51-byte PLY vertex with normals (d2pc_format.h compiled for the host) against the oracle, and the
argument validation of the new C entry points (nothing is launched)."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import d2pc_normals_oracle as N
from oracle import d2pc_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _angle(a, b):
    """unsigned angle between the lines spanned by a and b (atan2: accurate near 0)"""
    return np.arctan2(np.linalg.norm(np.cross(a, b), axis=1), np.abs((a * b).sum(1)))


def _brute_neighbours(p, k, radius=None):
    P = p.astype(np.float64)
    d = P[:, None, :] - P[None, :, :]
    d2 = d[..., 0] * d[..., 0]
    d2 = d2 + d[..., 1] * d[..., 1]
    d2 = d2 + d[..., 2] * d[..., 2]
    n = len(p)
    order = np.lexsort((np.broadcast_to(np.arange(n), (n, n)), d2), axis=1)[:, :min(k, n)]
    r2 = radius * radius if radius else np.inf
    return [o[d2[i, o] < r2] for i, o in enumerate(order)]


def test_fast_eigen_matches_eigh():
    rng = np.random.default_rng(0)
    M = rng.standard_normal((20000, 3, 3))
    S = M @ np.transpose(M, (0, 2, 1)) * 10.0 ** rng.uniform(-6, 6, (20000, 1, 1))
    Q, _ = np.linalg.qr(rng.standard_normal((20000, 3, 3)))
    lam = np.sort(rng.random((20000, 3)), 1)
    lam[:5000, 1] = lam[:5000, 0] * (1 + 10.0 ** rng.uniform(-8, -1, 5000))   # nearly coalescing pairs
    lam[5000:6000, 0] = 0.0                                                     # rank 2: plane covariances
    S = np.concatenate([S, Q @ (lam[:, :, None] * np.transpose(Q, (0, 2, 1)))])
    S = (S + np.transpose(S, (0, 2, 1))) / 2
    v = N.fast_eigen3x3(S[:, [0, 0, 0, 1, 1, 2], [0, 1, 2, 1, 2, 2]])
    assert np.allclose(np.linalg.norm(v, axis=1), 1.0, atol=1e-12)
    w, V = np.linalg.eigh(S)
    relgap = (w[:, 1] - w[:, 0]) / w[:, 2]
    ang = _angle(v, V[:, :, 0])
    # the closed-form eigenvalues lose accuracy as the two smallest coalesce: error ~ 1e-9 / relative gap
    assert (ang * relgap).max() < 1e-7
    assert ang[relgap > 1e-3].max() < 1e-9


def test_fast_eigen_degenerate_branches():
    z = N.fast_eigen3x3(np.zeros((1, 6)))
    assert (z == 0).all()
    diag = N.fast_eigen3x3(np.array([[3.0, 0, 0, 1.0, 0, 2.0], [1.0, 0, 0, 1.0, 0, 2.0], [1.0, 0, 0, 1.0, 0, 1.0],
                                     [2.0, 0, 0, 3.0, 0, 1.0]]))
    assert diag.tolist() == [[0, 1, 0], [0, 0, 1], [0, 0, 1], [0, 0, 1]]   # strictly smallest, else z


def test_planes_and_lines_give_analytic_normals():
    rng = np.random.default_rng(1)
    uv = rng.random((3000, 2)) * 4
    # z = 2 plane: (0, 0, 1) up to sign; oriented to the camera at the origin -> (0, 0, -1)
    p = np.c_[uv, np.full(3000, 2.0)].astype(np.float32)
    n = N.estimate_normals(p)
    assert np.allclose(n, [0, 0, -1], atol=1e-12)
    # tilted plane through the origin offset along its normal
    a = np.array([1.0, -2.0, 2.0]) / 3.0
    e1 = np.cross(a, [1.0, 0, 0]); e1 /= np.linalg.norm(e1)
    e2 = np.cross(a, e1)
    p = (uv[:, :1] * e1 + uv[:, 1:] * e2 + 5.0 * a).astype(np.float32)
    n = N.estimate_normals(p, knn=20)
    assert _angle(n, np.broadcast_to(a, n.shape)).max() < 1e-5     # float32 coordinates
    assert ((n * (-p.astype(np.float64))).sum(1) >= 0).all()
    # a line: every normal is perpendicular to it
    t = rng.random(500)
    d = np.array([7.0, -3.0, 0.5])
    p = (t[:, None] * d + [1.0, 2.0, 3.0]).astype(np.float32)
    n = N.estimate_normals(p, knn=10)
    assert np.abs(n @ (d / np.linalg.norm(d))).max() < 1e-5
    assert np.allclose(np.linalg.norm(n, axis=1), 1.0)


def test_small_neighbourhoods_give_z():
    rng = np.random.default_rng(2)
    for n in (1, 2):
        p = rng.standard_normal((n, 3)).astype(np.float32)
        out, cov = N.estimate_normals(p, orient_towards=None, return_covariances=True)
        assert out.tolist() == [[0.0, 0.0, 1.0]] * n and (cov == [1, 0, 0, 1, 0, 1]).all()
    p = rng.standard_normal((200, 3)).astype(np.float32)
    for k in (1, 2):
        assert (N.estimate_normals(p, knn=k, orient_towards=None) == [0, 0, 1]).all()
        assert (np.abs(N.estimate_normals(p, knn=k)) == [0, 0, 1]).all()
    # a radius smaller than any spacing: every point has only itself
    g = np.stack(np.meshgrid(*[np.arange(5)] * 3, indexing="ij"), -1).reshape(-1, 3).astype(np.float32)
    assert (N.estimate_normals(g, radius=0.5, orient_towards=None) == [0, 0, 1]).all()
    # exactly the spacing: the strict d2 < r^2 still leaves each point alone
    assert (N.estimate_normals(g, radius=1.0, orient_towards=None) == [0, 0, 1]).all()
    # just above it: interior points see their 6 neighbours
    cov = N.estimate_normals(g, radius=1.0000001, orient_towards=None, return_covariances=True)[1]
    assert not (cov == [1, 0, 0, 1, 0, 1]).all(axis=1).any()


def test_neighbours_equal_brute_force_with_ties():
    rng = np.random.default_rng(3)
    lattice = (np.stack(np.meshgrid(*[np.arange(7)] * 3, indexing="ij"), -1).reshape(-1, 3) * 0.25).astype(np.float32)
    dup = np.repeat(rng.random((40, 3)).astype(np.float32), 9, axis=0)
    blob = rng.standard_normal((500, 3)).astype(np.float32)
    for p in (lattice, dup, blob):
        for k, radius in ((1, None), (3, None), (30, None), (64, None), (30, 0.3), (20, 0.26), (64, 1.0)):
            rows, valid = N.neighbours(p, k, radius)
            want = _brute_neighbours(p, k, radius)
            for i in range(len(p)):
                assert np.array_equal(rows[i][valid[i]], want[i]), (len(p), k, radius, i)
                assert valid[i][:len(want[i])].all() and not valid[i][len(want[i]):].any()


def test_orientation_and_refusals():
    rng = np.random.default_rng(4)
    p = rng.standard_normal((1000, 3)).astype(np.float32)
    c = np.array([0.5, -3.0, 9.0])
    n = N.estimate_normals(p, orient_towards=c)
    assert ((n * (c - p.astype(np.float64))).sum(1) >= 0).all()
    raw = N.estimate_normals(p, orient_towards=None)
    assert (np.abs(raw) == np.abs(n)).all()
    bad = p.copy()
    bad[3, 1] = np.nan
    with pytest.raises(ValueError):
        N.estimate_normals(bad)
    bad[3, 1] = np.inf
    with pytest.raises(ValueError):
        N.estimate_normals(bad)


def test_ply_normal_layout_and_header():
    from image_to_pointcloud_b200 import writers
    assert N.PLY_NORMAL_RECORD_DTYPE.itemsize == writers.PLY_NORMAL_RECORD_BYTES == 51
    assert writers.PLY_NORMAL_HEADER == N.PLY_NORMAL_HEADER
    props = [ln.split()[-1] for ln in N.PLY_NORMAL_HEADER.splitlines() if ln.startswith("property")]
    assert props == list(N.PLY_NORMAL_RECORD_DTYPE.names) == ["x", "y", "z", "nx", "ny", "nz", "red", "green", "blue"]
    # without normals the header is the one written today
    assert writers.PLY_HEADER == O.PLY_HEADER


HOST_SRC = r"""
#include "d2pc_format.h"
extern "C" void ply_normals(const float *xyz, const double *nrm, const float *rgb, long n, unsigned char *out) {
  for (long i = 0; i < n; ++i) d2pc::ply_normal_record(xyz + 3 * i, nrm + 3 * i, rgb + 3 * i, out + 51 * i);
}
"""


def test_ply_normal_records_host_build_equal_oracle(tmp_path):
    """The device's record writer (d2pc_format.h) compiled for the host produces the oracle's bytes."""
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    src = tmp_path / "plyn.cpp"
    src.write_text(HOST_SRC)
    so = tmp_path / "plyn.so"
    res = subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off",
                          "-I", os.path.join(ROOT, "image_to_pointcloud_b200", "csrc"), str(src), "-o", str(so)],
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    lib = C.CDLL(str(so))
    from tests import cases
    p, c = cases.writer_rows(11, 3000)
    c[:8, 0] = [-5.0, 300.0, np.nan, 0.4, 0.5, 254.5, 127.5, 1e9]
    rng = np.random.default_rng(5)
    nrm = rng.standard_normal((3000, 3))
    nrm[:6] = [[0.0, 0.0, 1.0], [-0.0, 0.0, -1.0], [np.nan, 0, 0], [1e-300, -1e300, 0], [5e-324, 1, 0], [1, 1, 1]]
    out = np.zeros((3000, 51), np.uint8)
    lib.ply_normals(p.ctypes.data, nrm.ctypes.data, c.ctypes.data, C.c_long(3000), out.ctypes.data)
    want = N.ply_normal_records(p, nrm, c)
    assert out.tobytes() == want.tobytes()


def test_c_entry_points_validate_arguments():
    import image_to_pointcloud_b200 as m
    lib = m.load_library()
    INVALID, SMALL = 1, 2
    nb = C.c_size_t(0)
    assert lib.d2pc_normals_scratch_bytes(0, C.byref(nb)) == INVALID
    assert lib.d2pc_normals_scratch_bytes(1000, None) == INVALID
    assert lib.d2pc_normals_scratch_bytes(1000, C.byref(nb)) == 0 and nb.value > 0
    fake = 0x7f0000000000   # never dereferenced: every call below fails validation before a launch
    cam = (C.c_double * 3)(0.0, 0.0, 0.0)

    def call(xyz=fake, count=fake, cap=1000, bounds=fake, knn=30, radius=0.0, orient=1, camera=cam, scratch=fake,
             sbytes=nb.value, out=fake, cov=None):
        return lib.d2pc_normals_enqueue(xyz, count, cap, bounds, knn, radius, orient, camera, scratch, sbytes, out,
                                        cov, None)
    for kw in (dict(xyz=None), dict(count=None), dict(bounds=None), dict(scratch=None), dict(out=None),
               dict(cap=0), dict(knn=0), dict(knn=65), dict(knn=-3), dict(radius=float("nan")), dict(camera=None),
               dict(camera=(C.c_double * 3)(0.0, float("inf"), 0.0)), dict(scratch=fake + 8)):
        assert call(**kw) == INVALID, kw
    assert call(sbytes=nb.value - 1) == SMALL
    assert lib.d2pc_ply_normal_records_enqueue(None, fake, fake, fake, 10, fake, None) == INVALID
    assert lib.d2pc_ply_normal_records_enqueue(fake, None, fake, fake, 10, fake, None) == INVALID
    assert lib.d2pc_ply_normal_records_enqueue(fake, fake, fake, fake, 0, fake, None) == INVALID
    assert lib.d2pc_ply_normal_records_enqueue(fake, fake, fake, fake, 10, fake + 4, None) == INVALID
