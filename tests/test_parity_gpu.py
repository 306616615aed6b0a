"""GPU (-m gpu): the CUDA path, called through the public API / C ABI, against the oracle and the
golden vectors of the unmodified reference.  Bit-exact for xyz, rgb, masks and voxel indices;
voxel means within 1e-5 relative (float64 atomics are order-dependent)."""
import hashlib
import os
import warnings

import numpy as np
import pytest

from oracle import d2pc_oracle as O
from tests import cases
from tests.conftest import GOLDEN_DIR, assert_bits_equal

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def m():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import image_to_pointcloud_b200 as mod
    mod.load_library()
    return mod


def _oracle(img, dep, **kw):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return O.depth_to_point_cloud(img, dep, **kw)


def test_small_goldens_bit_exact(m, small_golden):
    n_run = 0
    for name in small_golden.names:
        img, dep, kw, pts, cols = small_golden.case(name)
        p, c = m.depth_to_point_cloud(img, dep, **kw)
        assert isinstance(p, np.ndarray) and p.dtype == np.float32 and p.flags["C_CONTIGUOUS"]
        if name == "smooth_minmax_f32":  # float32 blur path of OpenCV/IPP is not bit-modelled
            np.testing.assert_allclose(p, pts, rtol=1e-5, atol=1e-6)
        else:
            assert_bits_equal(p, pts, f"{name} points")
        assert_bits_equal(c, cols, f"{name} colors")
        n_run += 1
    assert n_run >= 32


@pytest.mark.parametrize("name", list(cases.LARGE_CASES))
def test_large_goldens_sha(m, large_golden, name):
    g = large_golden["cases"][name]
    img, dep, kw = cases.build_case(cases.LARGE_CASES[name])
    p, c = m.depth_to_point_cloud(img, dep, **kw)
    assert len(p) == g["n_points"]
    s = g["sample_stride"]
    assert p[::s].tobytes().hex() == g["points_sample_hex"], "sampled rows differ from the reference"
    assert hashlib.sha256(p.tobytes()).hexdigest() == g["points_sha256"]
    assert hashlib.sha256(c.tobytes()).hexdigest() == g["colors_sha256"]


def _engine_run(m, imgs, deps, **kw):
    import torch
    force = kw.pop("force_fallback", False)
    B = len(imgs)
    H, W = imgs[0].shape[:2]
    h, w = deps[0].shape[:2]
    eng = m.FrameEngine(H, W, h, w, batch=B, img_c=3)
    cfg = eng.make_config(force_fallback=force, **kw)
    d = torch.from_numpy(np.stack(deps)).cuda()
    i = torch.from_numpy(np.stack(imgs)).cuda()
    res = eng.process(cfg, d, i)
    return eng, cfg, res


def test_fallback_path_equals_fast_path_and_oracle(m):
    """The exact radix-select fallback and the sampled fast path are independent selections:
    both must give the oracle's percentiles and points."""
    rng = np.random.default_rng(31)
    imgs = [rng.integers(0, 256, (120, 200, 3), dtype=np.uint8) for _ in range(4)]
    deps = [(rng.random((120, 200)) * 20).astype(np.float32),
            np.round(rng.random((120, 200)) * 20).astype(np.float32),
            (rng.standard_normal((120, 200)) * 50).astype(np.float32),
            np.exp(rng.standard_normal((120, 200)) * 3).astype(np.float32)]
    outs = {}
    for force in (False, True):
        eng, cfg, res = _engine_run(m, imgs, deps, density="high", force_fallback=force)
        prm = eng.frame_params(cfg)
        outs[force] = (res.xyz.cpu().numpy(), res.rgb.cpu().numpy(), prm)
        for b in range(4):
            po, co, info = O.depth_to_point_cloud(imgs[b], deps[b], density="high", return_info=True)
            assert prm[b]["status"] == 1
            assert np.float64(prm[b]["p2"]).tobytes() == np.float64(info["p2"]).tobytes(), (force, b)
            assert np.float64(prm[b]["p98"]).tobytes() == np.float64(info["p98"]).tobytes(), (force, b)
            assert_bits_equal(outs[force][0][b], po, f"force={force} frame {b}")
            assert_bits_equal(outs[force][1][b], co, f"force={force} frame {b}")
    assert outs[False][2][0]["reserved"][0] == 0, "fast path should not have failed on uniform data"


def test_batch_with_mixed_frames(m):
    """One batch: clean frame, NaN/inf frame (fallback), constant frame (zeros branch), two-outlier
    frame (min/max branch), heavy-tie frame.  Each frame must match the oracle on its own."""
    rng = np.random.default_rng(32)
    H, W = 96, 160
    imgs = [rng.integers(0, 256, (H, W, 3), dtype=np.uint8) for _ in range(5)]
    deps = [cases.make_depth(H, W, 1, "uniform"), cases.make_depth(H, W, 2, "nonfinite"),
            cases.make_depth(H, W, 3, "constant"), cases.make_depth(H, W, 4, "two_outliers"),
            cases.make_depth(H, W, 5, "ties")]
    for kw in (dict(density="high"), dict(density="medium", invert=False, depth_scale=3.5)):
        eng, cfg, res = _engine_run(m, imgs, deps, **kw)
        prm = eng.frame_params(cfg)
        assert [p["branch"] for p in prm] == [0, 0, 2, 1, 0]
        assert prm[1]["n_nonfinite"] > 0
        for b in range(5):
            po, co = _oracle(imgs[b], deps[b], **kw)
            assert int(res.count[b]) == len(po)
            assert_bits_equal(res.xyz[b].cpu().numpy(), po, f"{kw} frame {b}")
            assert_bits_equal(res.rgb[b].cpu().numpy(), co, f"{kw} frame {b}")


def test_resized_batch_all_strides(m):
    rng = np.random.default_rng(33)
    H, W, h, w = 121, 161, 77, 91
    imgs = [rng.integers(0, 256, (H, W, 3), dtype=np.uint8) for _ in range(3)]
    deps = [(rng.random((h, w)) * 20).astype(np.float32) for _ in range(3)]
    deps[1][5, 5] = np.nan
    deps[1][0, 0] = np.inf  # corner tap: IPP turns it into NaN
    for dens in ("low", "medium", "high"):
        eng, cfg, res = _engine_run(m, imgs, deps, density=dens)
        for b in range(3):
            po, co = _oracle(imgs[b], deps[b], density=dens)
            assert_bits_equal(res.xyz[b].cpu().numpy(), po, f"{dens} frame {b}")
            assert_bits_equal(res.rgb[b].cpu().numpy(), co, f"{dens} frame {b}")


def test_float64_depth_that_needs_a_resize_is_cast_first(m):
    """Documented deviation (api.check_depth_dtype): a float64 map is cast to float32 and then interpolated like
    a float32 map (bit-exact against the oracle on the cast map); the reference would interpolate in float64 --
    the result stays inside the 1e-5 tolerance of that."""
    rng = np.random.default_rng(5)
    img = rng.integers(0, 256, (90, 120, 3), dtype=np.uint8)
    dep = rng.random((41, 57)) * 20
    p, c = m.depth_to_point_cloud(img, dep, density="high")
    po, co = _oracle(img, dep.astype(np.float32), density="high")
    assert_bits_equal(p, po, "float64 depth")
    assert_bits_equal(c, co, "float64 depth")
    try:
        import cv2
    except ImportError:
        return
    # what the reference does: interpolate in float64, cast afterwards; then its own float32 pipeline
    d64 = cv2.resize(dep, (120, 90), interpolation=cv2.INTER_LINEAR).astype(np.float32)
    pr, _ = _oracle(img, d64, density="high")
    assert np.allclose(p, pr, rtol=1e-5, atol=1e-5)


def test_resized_tiled_scan_geometries(m):
    """Widths that are a multiple of 4 take the shared-memory tiled resize (up- and mild down-scaling);
    strong down-scaling falls back to the direct kernel.  Non-finite values sit on corners and edges."""
    rng = np.random.default_rng(41)
    for (H, W, h, w) in [(200, 320, 77, 91), (96, 160, 100, 170), (130, 256, 37, 300), (64, 132, 200, 260),
                         (33, 4, 10, 3), (480, 640, 518, 686)]:
        img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        deps = [(rng.random((h, w)) * 20).astype(np.float32) for _ in range(2)]
        deps[1][0, 0] = np.inf
        deps[1][h - 1, w - 1] = -np.inf
        deps[1][0, w // 2] = np.nan
        deps[1][h // 2, 0] = np.inf
        eng, cfg, res = _engine_run(m, [img, img], deps, density="high")
        for b in range(2):
            po, co = _oracle(img, deps[b], density="high")
            assert_bits_equal(res.xyz[b].cpu().numpy(), po, f"{(H, W, h, w)} frame {b}")
        po, co = _oracle(img, deps[0], density="medium", invert=False)
        p, c = m.depth_to_point_cloud(img, deps[0], density="medium", invert=False, z_range=(1.0, 9.0))
        keep = O.range_mask(po, 1.0, 9.0)
        assert_bits_equal(p, po[keep], f"{(H, W, h, w)} masked medium")


def test_strided_fast_emit(m):
    """density medium / low on widths that are multiples of 8 / 16 take the vectorised strided path;
    other widths the generic one.  Both must match the oracle bit for bit (incl. the fused bounds)."""
    rng = np.random.default_rng(42)
    for (H, W, h, w) in [(120, 320, 120, 320), (121, 336, 60, 100), (64, 1040, 64, 1040), (50, 24, 50, 24),
                         (37, 48, 37, 48)]:
        img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        dep = (rng.random((h, w)) * 20).astype(np.float32)
        for dens in ("medium", "low"):
            for inv in (True, False):
                po, co = _oracle(img, dep, density=dens, invert=inv)
                p, c, bd = m.depth_to_point_cloud(img, dep, density=dens, invert=inv, return_bounds=True)
                assert_bits_equal(p, po, f"{(H, W)} {dens} invert={inv}")
                assert_bits_equal(c, co, f"{(H, W)} {dens} colours")
                assert bd["minX"] == float(po[:, 0].min()) and bd["maxZ"] == float(po[:, 2].max())
                p, c = m.depth_to_point_cloud(img, dep, density=dens, invert=inv)
                assert_bits_equal(p, po, f"{(H, W)} {dens} invert={inv} (no bounds)")
                assert_bits_equal(c, co, f"{(H, W)} {dens} colours (no bounds)")


def test_percentile_selection_on_hard_distributions(m):
    """Exact order statistics for sizes above the sampling threshold, incl. ReLU-style zeros."""
    rng = np.random.default_rng(34)
    H, W = 360, 640
    img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    variants = {
        "uniform": (rng.random((H, W)) * 20).astype(np.float32),
        "relu_zeros_30pct": np.maximum(rng.standard_normal((H, W)) - 0.5, 0).astype(np.float32),
        "narrow": (10 + rng.random((H, W)) * 1e-3).astype(np.float32),
        "quantised": np.round(rng.random((H, W)) * 50).astype(np.float32),
        "lognormal": np.exp(rng.standard_normal((H, W)) * 4).astype(np.float32),
        "negative": (-np.exp(rng.standard_normal((H, W)))).astype(np.float32),
        "sorted_ramp": np.linspace(0, 1, H * W, dtype=np.float32).reshape(H, W),
        "periodic": np.tile(np.arange(W, dtype=np.float32) % 27, (H, 1)),
    }
    for name, dep in variants.items():
        eng, cfg, res = _engine_run(m, [img], [dep], density="medium")
        prm = eng.frame_params(cfg)[0]
        po, co, info = O.depth_to_point_cloud(img, dep, density="medium", return_info=True)
        assert np.float64(prm["p2"]).tobytes() == np.float64(info["p2"]).tobytes(), name
        assert np.float64(prm["p98"]).tobytes() == np.float64(info["p98"]).tobytes(), name
        assert_bits_equal(res.xyz[0].cpu().numpy(), po, name)


def test_cooperative_selection_equals_single_cta_selection(m, monkeypatch):
    """The K-CTA two-launch selection (small batches, 4K frames) against the one-CTA-per-bracket kernel and the
    oracle: p2 / p98 float64 bit-equal for every K, on batches of 3 and 5 frames (batches of 1 or 2 take the
    index-ordered kernel) with hard distributions and a frame that needs the fallback."""
    rng = np.random.default_rng(52)
    H, W = 270, 480
    deps = [
        (rng.random((H, W)) * 20).astype(np.float32),
        np.maximum(rng.standard_normal((H, W)) - 0.5, 0).astype(np.float32),      # 30% exact zeros
        np.round(rng.random((H, W)) * 50).astype(np.float32),                      # heavy ties
        (10 + rng.random((H, W)) * 1e-3).astype(np.float32),                       # narrow key range
        np.exp(rng.standard_normal((H, W)) * 4).astype(np.float32),
    ]
    deps[4][11, 13] = np.nan                                                        # exact fallback
    imgs = [rng.integers(0, 256, (H, W, 3), dtype=np.uint8) for _ in deps]
    want = [O.depth_to_point_cloud(i, d, density="low", return_info=True) for i, d in zip(imgs, deps)]
    for nb in (3, 5):
        for K in ("0", "2", "3", "8", "64"):
            monkeypatch.setenv("D2PC_SELECT_COOP", K)
            eng, cfg, res = _engine_run(m, imgs[:nb], deps[:nb], density="low")
            prm = eng.frame_params(cfg)
            for b in range(nb):
                po, co, info = want[b]
                assert np.float64(prm[b]["p2"]).tobytes() == np.float64(info["p2"]).tobytes(), (nb, K, b)
                assert np.float64(prm[b]["p98"]).tobytes() == np.float64(info["p98"]).tobytes(), (nb, K, b)
                assert_bits_equal(res.xyz[b].cpu().numpy(), po, f"nb={nb} K={K} frame {b}")


def test_multi_tile_scan_equals_single_tile_scan(m, monkeypatch):
    """The scan kernel that walks several tiles per CTA (large grids; forced here with D2PC_SCAN_TPC) against the
    oracle: frames whose last tile is partial, tile counts that leave a CTA with fewer tiles than TPC, clustered
    tiles (every pixel of a tile deferred), a frame for the fallback."""
    rng = np.random.default_rng(54)

    def frames(H, W):
        deps = [
            (rng.random((H, W)) * 20).astype(np.float32),
            np.sort((rng.random(H * W) * 20).astype(np.float32)).reshape(H, W),   # extremes clustered in whole tiles
            np.round(rng.random((H, W)) * 50).astype(np.float32),
            (rng.random((H, W)) * 20).astype(np.float32),
        ]
        deps[3][H // 2, W // 2] = np.inf
        imgs = [rng.integers(0, 256, (H, W, 3), dtype=np.uint8) for _ in deps]
        want = [O.depth_to_point_cloud(i, d, density="medium", return_info=True) for i, d in zip(imgs, deps)]
        return imgs, deps, want

    # 203 x 517 = 104 951 pixels: 12 full tiles + a partial one, unaligned rows; 256 x 512: 16 full tiles
    cases_ = [frames(203, 517), frames(256, 512)]
    for tpc in ("1", "2", "4"):
        monkeypatch.setenv("D2PC_SCAN_TPC", tpc)
        for imgs, deps, want in cases_:
            eng, cfg, res = _engine_run(m, imgs, deps, density="medium")
            prm = eng.frame_params(cfg)
            for b, (po, co, info) in enumerate(want):
                assert np.float64(prm[b]["p2"]).tobytes() == np.float64(info["p2"]).tobytes(), (tpc, deps[0].shape, b)
                assert np.float64(prm[b]["p98"]).tobytes() == np.float64(info["p98"]).tobytes(), (tpc, deps[0].shape, b)
                assert_bits_equal(res.xyz[b].cpu().numpy(), po, f"tpc={tpc} {deps[0].shape} frame {b}")


def test_range_mask_and_compaction(m):
    rng = np.random.default_rng(35)
    for (H, W, h, w) in [(96, 160, 96, 160), (121, 161, 77, 91), (300, 500, 300, 500)]:
        img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        dep = (rng.random((h, w)) * 20).astype(np.float32)
        dep[3, 4] = np.nan
        for dens in ("high", "medium"):
            for zr in ((0.5, 9.5), (2.0, 2.5), (20.0, 30.0), (0.0, 10.0)):
                po, co = _oracle(img, dep, density=dens)
                keep = O.range_mask(po, *zr)
                p, c = m.depth_to_point_cloud(img, dep, density=dens, z_range=zr)
                assert len(p) == int(keep.sum()), (H, W, dens, zr)
                assert_bits_equal(p, po[keep], f"mask {zr} points")   # raster order preserved
                assert_bits_equal(c, co[keep], f"mask {zr} colors")
    # drop_nonfinite drops the repaired pixels
    po, co = _oracle(img, dep, density="high")
    p, c = m.depth_to_point_cloud(img, dep, density="high", drop_nonfinite=True)
    fin = np.isfinite(dep).ravel()
    assert_bits_equal(p, po[fin], "drop_nonfinite")


def test_range_mask_with_whole_tiles_kept_or_dropped(m):
    """Coherent masks: emit tiles (1024 consecutive rows) that keep nothing, everything (at 16-byte aligned and
    at unaligned destinations) or a part, in every order."""
    rng = np.random.default_rng(37)
    H, W = 48, 1024   # one tile per image row
    img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    base = np.repeat(np.linspace(1.0, 19.0, H, dtype=np.float32)[:, None], W, axis=1)
    base[::5] = 15.0                                     # rows jumping in and out of the range
    dep = (base + rng.random((H, W)).astype(np.float32) * 0.01).astype(np.float32)
    dep[7, :3] = 19.5; dep[20, 500] = 0.5; dep[33, 1023] = 19.9   # partial tiles shift the alignment of later ones
    for inv in (True, False):
        for zr in ((3.0, 7.0), (0.0, 10.0), (4.0, 4.5), (9.9, 10.0)):
            po, co = _oracle(img, dep, density="high", invert=inv)
            keep = O.range_mask(po, *zr)
            p, c = m.depth_to_point_cloud(img, dep, density="high", invert=inv, z_range=zr)
            assert len(p) == int(keep.sum()), (inv, zr)
            assert_bits_equal(p, po[keep], f"tiles {inv} {zr} points")
            assert_bits_equal(c, co[keep], f"tiles {inv} {zr} colors")
            pb, cb, bnd = m.depth_to_point_cloud(img, dep, density="high", invert=inv, z_range=zr, return_bounds=True)
            assert_bits_equal(pb, po[keep], "tiles + bounds")
            if len(pb):
                assert bnd["minX"] == float(pb[:, 0].min()) and bnd["maxZ"] == float(pb[:, 2].max())


def test_voxel_downsample(m):
    rng = np.random.default_rng(36)
    H, W = 240, 320
    img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    dep = cases.make_depth(H, W, 9, "scene")
    for vs in (0.05, 0.5, 0.005):
        for zr in (None, (0.5, 9.5)):
            po, co = _oracle(img, dep, density="high")
            if zr is not None:
                po, co, _ = O.apply_range_mask(po, co, *zr)
            vp, vc, vidx = O.voxel_downsample(po, co, vs)
            p, c, idx = m.depth_to_point_cloud(img, dep, density="high", z_range=zr, voxel_size=vs,
                                               return_voxel_index=True)
            assert len(p) == len(vp), (vs, zr)
            key = (idx[:, 0].astype(np.int64) << 42) | (idx[:, 1].astype(np.int64) << 21) | idx[:, 2]
            order = np.argsort(key)
            assert np.array_equal(idx[order], vidx), "voxel indices must be bit-exact"
            np.testing.assert_allclose(p[order], vp, rtol=1e-5, atol=1e-6)
            np.testing.assert_allclose(c[order], vc, rtol=1e-6, atol=0)   # integer colour sums are exact
            # fixed-point coordinate sums: deterministic, same bits on a second run (order-normalised)
            p2, c2, idx2 = m.depth_to_point_cloud(img, dep, density="high", z_range=zr, voxel_size=vs,
                                                  return_voxel_index=True)
            key2 = (idx2[:, 0].astype(np.int64) << 42) | (idx2[:, 1].astype(np.int64) << 21) | idx2[:, 2]
            o2 = np.argsort(key2)
            assert np.array_equal(p[order].view(np.uint32), p2[o2].view(np.uint32))
            assert np.array_equal(c[order].view(np.uint32), c2[o2].view(np.uint32))
    with pytest.raises(ValueError):
        m.depth_to_point_cloud(img, dep, density="high", voxel_size=1e-9)
    # a mask that keeps nothing: empty voxel output, no error
    p, c, idx = m.depth_to_point_cloud(img, dep, density="high", z_range=(20.0, 30.0), voxel_size=0.05, return_voxel_index=True)
    assert p.shape == (0, 3) and c.shape == (0, 3) and idx.shape == (0, 3)


def test_smoothing_larger_frames(m):
    """a6 at sizes with W % 4 != 0 (scalar tail of OpenCV's row filter), with strides and a mask."""
    rng = np.random.default_rng(38)
    for (H, W, h, w) in [(121, 161, 77, 91), (96, 160, 96, 160), (50, 47, 50, 47)]:
        img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        dep = (rng.random((h, w)) * 20).astype(np.float32)
        for kw in (dict(density="high", smooth=True), dict(density="medium", smooth=True, smooth_ksize=7, invert=False),
                   dict(density="low", smooth=True, smooth_ksize=9)):
            po, co = _oracle(img, dep, **kw)
            p, c = m.depth_to_point_cloud(img, dep, **kw)
            assert_bits_equal(p, po, f"smooth {H}x{W} {kw}")
            assert_bits_equal(c, co, f"smooth {H}x{W} {kw}")
        po, co = _oracle(img, dep, density="high", smooth=True)
        keep = O.range_mask(po, 2.0, 8.0)
        p, c = m.depth_to_point_cloud(img, dep, density="high", smooth=True, z_range=(2.0, 8.0))
        assert_bits_equal(p, po[keep], "smooth + mask")


def test_smoothing_with_large_kernels(m):
    """a6 with kernels far beyond the caller's default 5 (the reference accepts any size, app.py:209-212): up to
    255 taps, larger than the image (REFLECT_101 wraps repeatedly).  Coefficients for k > 7 come from exp(): within
    the 1e-5 tolerance of the oracle (which equals cv2.GaussianBlur to 1e-15), not bit-pinned."""
    rng = np.random.default_rng(53)
    H, W = 70, 90
    img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    dep = (rng.random((H, W)) * 20).astype(np.float32)
    for k in (33, 63, 255):
        po, co = _oracle(img, dep, density="medium", smooth=True, smooth_ksize=k)
        p, c = m.depth_to_point_cloud(img, dep, density="medium", smooth=True, smooth_ksize=k)
        assert p.shape == po.shape and np.array_equal(c, co)
        np.testing.assert_allclose(p, po, rtol=1e-5, atol=1e-6, err_msg=f"k={k}")
    with pytest.raises(ValueError):   # beyond the coefficient table: refused before any GPU work
        m.depth_to_point_cloud(img, dep, smooth=True, smooth_ksize=257)


def test_bounds_equal_numpy_minmax(m):
    """f4: the bounds fused into emit equal points[:, k].min()/max() (generate_gis_metadata, app.py:393-400)."""
    rng = np.random.default_rng(39)
    for (H, W, h, w, kw) in [(96, 160, 96, 160, dict(density="high")), (121, 161, 77, 91, dict(density="medium")),
                             (96, 160, 96, 160, dict(density="high", z_range=(2.0, 8.0)))]:
        img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        dep = (rng.random((h, w)) * 20).astype(np.float32)
        p, c, b = m.depth_to_point_cloud(img, dep, return_bounds=True, **kw)
        want = {"minX": float(p[:, 0].min()), "maxX": float(p[:, 0].max()), "minY": float(p[:, 1].min()),
                "maxY": float(p[:, 1].max()), "minZ": float(p[:, 2].min()), "maxZ": float(p[:, 2].max())}
        assert b == want


def test_depth_preview(m, small_golden):
    """f2: colour-mapped preview bit-exact against the oracle; data URL equal to the reference's."""
    import json
    lut = np.load(os.path.join(GOLDEN_DIR, "plasma_lut_bgr.npy"))
    for name in json.loads(str(small_golden.z["__preview_names__"])):
        dep = small_golden.z[f"{name}/depth"]
        inv = bool(small_golden.z[f"{name}/invert"])
        got = m.depth_preview_bgr(dep, invert=inv)
        assert np.array_equal(got, O.depth_preview_bgr(dep, inv, lut)), name
        assert m.create_depth_preview(dep, invert=inv) == str(small_golden.z[f"{name}/data_url"]), name
    rng = np.random.default_rng(40)
    for shape in [(518, 686), (200, 333)]:
        dep = (rng.random(shape) * 20).astype(np.float32)
        dep[3, 3] = np.nan
        for inv in (True, False):
            assert np.array_equal(m.depth_preview_bgr(dep, invert=inv), O.depth_preview_bgr(dep, inv, lut))


def test_host_pipeline_matches_single_calls(m):
    rng = np.random.default_rng(37)
    H, W = 120, 200
    n = 11
    imgs = [rng.integers(0, 256, (H, W, 3), dtype=np.uint8) for _ in range(n)]
    deps = [(rng.random((H, W)) * (5 + i)).astype(np.float32) for i in range(n)]
    deps[4][7, 7] = np.inf
    outs = m.depth_to_point_cloud_batch(imgs, deps, density="high", chunk=4)
    assert len(outs) == n
    for i in range(n):
        po, co = _oracle(imgs[i], deps[i], density="high")
        assert_bits_equal(outs[i][0], po, f"frame {i}")
        assert_bits_equal(outs[i][1], co, f"frame {i}")
    outs = m.depth_to_point_cloud_batch(imgs[:3], deps[:3], density="medium", z_range=(1.0, 8.0), chunk=8)
    for i in range(3):
        po, co = _oracle(imgs[i], deps[i], density="medium")
        keep = O.range_mask(po, 1.0, 8.0)
        assert_bits_equal(outs[i][0], po[keep], f"masked frame {i}")


def test_multi_gpu_pipeline_shards_frames(m):
    """MultiGpuPipeline: one host thread per device pipeline, frames sharded by frame, no collective.  On a
    one-GPU box two pipelines on the same device exercise the same threading; with more GPUs every device runs."""
    import torch
    rng = np.random.default_rng(41)
    H, W, h, w, n = 96, 128, 41, 57, 13
    imgs = [rng.integers(0, 256, (H, W, 3), dtype=np.uint8) for _ in range(n)]
    deps = [(rng.random((h, w)) * (3 + i)).astype(np.float32) for i in range(n)]
    deps[5][2, 2] = np.nan   # one frame through the exact fallback
    devs = list(range(torch.cuda.device_count()))
    for devices in ([0, 0], devs if len(devs) > 1 else [0]):
        pipe = m.MultiGpuPipeline(H, W, h, w, devices=devices, chunk=4, density="medium")
        assert [len(r) for r in pipe.shards(n)] == [len(m.shard_frames(n, len(devices), r)) for r in range(len(devices))]
        outs = pipe.run(imgs, deps)
        assert len(outs) == n
        for i in range(n):
            po, co = _oracle(imgs[i], deps[i], density="medium")
            assert_bits_equal(outs[i][0], po, f"frame {i} on {devices}")
            assert_bits_equal(outs[i][1], co, f"frame {i} on {devices}")


def test_4k_full_size_properties_and_oracle(m):
    """BASELINE config 3 size: full compare against the oracle plus size-independent properties."""
    img, dep, kw = cases.build_case(cases.LARGE_CASES["c3_4k_dav2"])
    p, c = m.depth_to_point_cloud(img, dep, **kw)
    assert p.shape == (2160 * 3840, 3)
    assert np.array_equal(c, img[:, :, ::-1].reshape(-1, 3).astype(np.float32))  # colour gather exact
    zmax = p[:, 2].max()
    assert 0.0 <= p[:, 2].min() and zmax <= 10.0
    assert p[1080 * 3840 + 1920, 0] == 0.0 and p[1080 * 3840 + 1920, 1] == 0.0  # u=cx, v=cy
    po, co = _oracle(img, dep, **kw)
    assert_bits_equal(p, po, "4K points")
    # idempotence: same input, same bits
    p2, _ = m.depth_to_point_cloud(img, dep, **kw)
    assert np.array_equal(p.view(np.uint32), p2.view(np.uint32))
