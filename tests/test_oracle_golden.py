"""CPU: the oracle (oracle/d2pc_oracle.py) against the committed golden vectors, which are
outputs of the UNMODIFIED reference function (backend/app.py:174-250) made by
oracle/make_golden.py.  This is what pins the oracle."""
import hashlib
import os
import warnings

import numpy as np
import pytest

from oracle import d2pc_oracle as O
from tests import cases
from tests.conftest import GOLDEN_DIR, assert_bits_equal


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def test_versions_pinned(small_golden, large_golden):
    import cv2
    # the reference's numerics depend on these (NEP 50 float64 chain, IPP bilinear)
    assert small_golden.versions["numpy"].split(".")[0] == np.__version__.split(".")[0] == "2"
    assert small_golden.versions["cv2"] == large_golden["versions"]["cv2"]
    assert small_golden.versions["ipp"] is True
    assert cv2.__version__  # importable; the oracle itself never calls cv2


def test_small_cases_bit_exact(small_golden):
    assert len(small_golden.names) >= 25
    for name in small_golden.names:
        img, dep, kw, pts, cols = small_golden.case(name)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            p, c = O.depth_to_point_cloud(img, dep, **kw)
        assert p.dtype == np.float32 and c.dtype == np.float32
        if name == "smooth_minmax_f32":  # float32 blur path of OpenCV/IPP is not bit-modelled
            np.testing.assert_allclose(p, pts, rtol=1e-5, atol=1e-6)
        else:
            assert_bits_equal(p, pts, f"{name} points")
        assert_bits_equal(c, cols, f"{name} colors")


def test_loop_restatement_matches_vectorised(small_golden):
    for name in ("up_medium_inv0", "odd_low", "minmax_fallback", "nonfinite_resized"):
        img, dep, kw, pts, cols = small_golden.case(name)
        p, c = O.depth_to_point_cloud_loop(img, dep, **kw)
        assert_bits_equal(p, pts, name)
        assert_bits_equal(c, cols, name)


@pytest.mark.parametrize("name", ["c1_480p_high", "c1_480p_medium", "c1_480p_low_noinv",
                                  "c2_1080p_native", "c2_1080p_dav2", "c2_1080p_scene_nonfinite"])
def test_large_cases_sha(large_golden, name):
    g = large_golden["cases"][name]
    img, dep, kw = cases.build_case(cases.LARGE_CASES[name])
    assert _sha(img) == g["image_sha256"] and _sha(dep) == g["depth_sha256"], "seeded inputs drifted"
    p, c = O.depth_to_point_cloud(img, dep, **kw)
    assert len(p) == g["n_points"]
    assert _sha(p) == g["points_sha256"]
    assert _sha(c) == g["colors_sha256"]
    s = g["sample_stride"]
    assert p[::s].tobytes().hex() == g["points_sample_hex"]


def test_analytic_known_answers():
    rng = np.random.default_rng(5)
    img = rng.integers(0, 256, (20, 30, 3), dtype=np.uint8)
    # constant map -> zeros branch -> every z = depth_scale when inverted
    p, c = O.depth_to_point_cloud(img, np.full((20, 30), 4.0, np.float32), density="high", depth_scale=7.0)
    assert np.all(p[:, 2] == np.float32(7.0))
    # centre pixel u = cx -> x = 0 ; v = cy -> y = 0
    W = 30
    assert p[10 * W + 15, 0] == 0.0 and p[10 * W + 15, 1] == 0.0
    # counts and colour gather for every stride
    for dens, s in O.DENSITY_STEP.items():
        p, c = O.depth_to_point_cloud(img, (rng.random((9, 11)) * 3).astype(np.float32), density=dens)
        assert len(p) == -(-20 // s) * -(-30 // s)
        assert np.array_equal(c, img[::s, ::s, ::-1].reshape(-1, 3).astype(np.float32))
    with pytest.raises(KeyError):
        O.depth_to_point_cloud(img, np.ones((20, 30), np.float32), density="ultra")


def test_percentile_restatement_matches_numpy():
    rng = np.random.default_rng(3)
    for t in range(200):
        n = int(rng.integers(1, 4000))
        d = (rng.standard_normal(n) * rng.choice([1e-3, 1.0, 1e4])).astype(np.float32)
        if t % 4 == 0:
            d = np.round(d) + np.float32(0.0)
            d[d == 0] = 0.0  # avoid -0/+0 ties, whose order numpy leaves unspecified
        a = np.percentile(d, [2, 98])
        b = O.percentiles_2_98(d)
        assert a[0].tobytes() == b[0].tobytes() and a[1].tobytes() == b[1].tobytes(), (n, a, b)


def test_nanmedian_restatement_matches_numpy():
    rng = np.random.default_rng(4)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for t in range(200):
            n = int(rng.integers(1, 100))
            d = rng.standard_normal(n).astype(np.float32)
            k = int(rng.integers(0, n + 1))
            idx = rng.choice(n, k, replace=False)
            d[idx] = rng.choice(np.array([np.nan, np.inf, -np.inf], np.float32), k)
            a, b = np.float32(np.nanmedian(d)), O.nanmedian_f32(d)
            assert a.tobytes() == b.tobytes() or (np.isnan(a) and np.isnan(b))


def test_resize_model_matches_cv2_here():
    """The IPP bilinear model against cv2.resize of this machine (skips if IPP is not active,
    e.g. on a CPU where OpenCV picks another code path)."""
    import cv2
    if not cv2.ipp.useIPP():
        pytest.skip("OpenCV without IPP: cv2.resize takes the generic path")
    rng = np.random.default_rng(6)
    shapes = [((518, 686), (480, 640)), ((37, 53), (48, 64)), ((48, 64), (37, 53)), ((2, 2), (9, 9)),
              ((100, 100), (33, 77)), ((7, 5), (121, 161)), ((300, 400), (300, 401)), ((96, 128), (48, 64))]
    for sh, dh in shapes:
        d = (rng.random(sh) * 20).astype(np.float32)
        a = cv2.resize(d, (dh[1], dh[0]), interpolation=cv2.INTER_LINEAR)
        b = O.resize_bilinear(d, dh[0], dh[1])
        assert O.count_bit_mismatch(a, b) == 0, (sh, dh)


def test_resize_model_for_one_pixel_sides_matches_cv2_here():
    """Sources with a 1-pixel side never reach IPP: OpenCV's own two-pass arithmetic (oracle
    _resize_bilinear_generic), with non-finite values in the way."""
    import cv2
    rng = np.random.default_rng(16)
    for t in range(120):
        sh = (1, int(rng.integers(1, 120))) if t % 2 else (int(rng.integers(1, 120)), 1)
        dh = (int(rng.integers(1, 160)), int(rng.integers(1, 160)))
        if sh == dh:
            continue
        d = (rng.standard_normal(sh) * 3).astype(np.float32)
        for _ in range(int(rng.integers(0, 3))):
            d.flat[rng.integers(d.size)] = (np.inf, -np.inf, np.nan)[int(rng.integers(3))]
        a = cv2.resize(d, (dh[1], dh[0]), interpolation=cv2.INTER_LINEAR)
        b = O.resize_bilinear(d, dh[0], dh[1])
        assert bool(np.all((a == b) | (np.isnan(a) & np.isnan(b)))), (sh, dh)


def test_fmaf_exact():
    rng = np.random.default_rng(8)
    a = rng.standard_normal(200000).astype(np.float32)
    b = rng.standard_normal(200000).astype(np.float32)
    c = (-(a.astype(np.float64) * b.astype(np.float64))).astype(np.float32)  # heavy cancellation
    got = O.fmaf(a, b, c)
    # exact reference with Python integers via fractions is slow; use longdouble + TwoSum-free check
    from fractions import Fraction
    for i in range(0, 200000, 997):
        exact = Fraction(float(a[i])) * Fraction(float(b[i])) + Fraction(float(c[i]))
        want = np.float32(float(exact)) if abs(exact) < 2 ** -1000 else None
        # float(Fraction) rounds correctly to float64; then emulate RN to float32 exactly:
        lo = np.float32(float(exact))
        cand = [np.nextafter(lo, np.float32(-np.inf)), lo, np.nextafter(lo, np.float32(np.inf))]
        best = min(cand, key=lambda x: (abs(Fraction(float(x)) - exact), int(np.float32(x).view(np.uint32)) & 1))
        assert got[i] == best, (i, a[i], b[i], c[i], got[i], best)


def test_depth_preview_oracle_matches_reference_data_urls(small_golden):
    """f2: the oracle's colour-mapped preview, PNG-encoded, equals the reference's data URL."""
    import base64
    import json

    import cv2
    lut = np.load(os.path.join(GOLDEN_DIR, "plasma_lut_bgr.npy"))
    names = json.loads(str(small_golden.z["__preview_names__"]))
    assert len(names) >= 3
    for name in names:
        dep = small_golden.z[f"{name}/depth"]
        inv = bool(small_golden.z[f"{name}/invert"])
        want = str(small_golden.z[f"{name}/data_url"])
        img = O.depth_preview_bgr(dep, inv, lut)
        ok, buf = cv2.imencode(".png", img)
        got = "data:image/png;base64," + base64.b64encode(buf.tobytes()).decode("utf-8")
        assert got == want, name
