"""GPU (-m gpu): the voxel grid (row ax-2, csrc/d2pc_voxel.cu) fed synthetic clouds built against it, straight
through FrameEngine.voxel_downsample, and through the stage at every density.  Reference: the oracle
(oracle.d2pc_oracle.voxel_downsample) and exact means (tests/voxel_cases.py).  The bar for every frame: the oracle's
voxels and indices bit-exact, colour means bit-exact, coordinate means within 2^-38 * E + ulp_f32(mean) (E = the
cloud's extent), and the same bits from a second run and from the split insert (D2PC_VOX_SPLIT=1)."""
import warnings

import numpy as np
import pytest

from oracle import d2pc_oracle as O
from tests import cases
from tests import voxel_cases as V

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def m():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import image_to_pointcloud_b200 as mod
    mod.load_library()
    return mod


@pytest.fixture(scope="module")
def engine(m):
    made = {}

    def get(H, W, B=1):
        if (H, W, B) not in made:
            made[(H, W, B)] = m.FrameEngine(H, W, batch=B)
        return made[(H, W, B)]
    yield get
    made.clear()


def _check(eng, cfg, frames, vs, what=""):
    """Fused insert against the reference; fused again and split: the same bits.  Returns the device frames."""
    got, vcount = V.run_device(eng, cfg, frames, vs)
    problems = []
    for b, ((p, c), g) in enumerate(zip(frames, got)):
        problems += V.check_frame(*g, p, c, vs, what=f"{what} frame {b}")[0]
    assert problems == [], problems[:4]
    assert len(vcount) == eng.batch and all(int(vcount[b]) == 0 for b in range(len(frames), eng.batch))
    for split in (False, True):
        again, _ = V.run_device(eng, cfg, frames, vs, split=split)
        for b, (g, a) in enumerate(zip(got, again)):
            assert V.canonical(*g) == V.canonical(*a), f"{what} frame {b}: {'split' if split else 'second'} run differs"
    return got


def _oracle_rows(img, dep, density, zr):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        po, co = O.depth_to_point_cloud(img, dep, density=density)
    if zr is not None:
        po, co, _ = O.apply_range_mask(po, co, *zr)
    return po, co


# ---- 1. voxel faces ---------------------------------------------------------------------------
@pytest.mark.parametrize("vs", [0.25, 0.1, 0.005, 1 / 3])
def test_points_on_and_next_to_voxel_faces(engine, vs):
    """floor(div_by_const_fast(p - vmin, vs)) against the oracle's IEEE division, at float32 points on the faces and
    up to 3 ulps either side, one axis per frame."""
    rng = np.random.default_rng(int(vs * 1e4))
    eng = engine(64, 96, 3)
    cfg = eng.make_config(want_bounds=True)
    for base in (0.0, -2.75, 13.1):
        frames = []
        for axis in range(3):
            p = V.face_cloud(vs, axis, rng, base=base)
            frames.append((p, V.colours(rng, len(p))))
        _check(eng, cfg, frames, vs, f"faces vs={vs} base={base}")


# ---- 2. index limit ---------------------------------------------------------------------------
@pytest.mark.parametrize("vs", [1.0, 0.005])
def test_index_limit(m, engine, vs):
    """A largest index of 2^21 - 1 (per axis, and on all three: all 63 key bits) is accepted and exact; 2^21 is
    refused with ValueError by the device and by the oracle."""
    rng = np.random.default_rng(21)
    eng = engine(64, 96, 1)
    cfg = eng.make_config(want_bounds=True)
    for axes in ((0,), (1,), (2,), (0, 1, 2)):
        p = V.limit_cloud(vs, axes, V.IDX_LIMIT - 1, rng)
        got = _check(eng, cfg, [(p, V.colours(rng, len(p)))], vs, f"limit axes={axes}")
        assert int(got[0][2][:, list(axes)].max()) == V.IDX_LIMIT - 1
        if axes == (0, 1, 2):
            assert int(V.pack_key(got[0][2]).max()) == (1 << 63) - 1
        q = V.limit_cloud(vs, axes, V.IDX_LIMIT, rng)
        c = V.colours(rng, len(q))
        with pytest.raises(ValueError):
            O.voxel_downsample(q, c, vs)
        with pytest.raises(ValueError):
            V.run_device(eng, cfg, [(q, c)], vs)
        # the refused frame leaves nothing behind: the next call on the same table is exact again
        _check(eng, cfg, [(p, V.colours(rng, len(p)))], vs, f"limit axes={axes} after a refusal")


# ---- 3. run structure of the segmented scan ----------------------------------------------------
def test_runs_across_groups_and_tiles(engine):
    rng = np.random.default_rng(3)
    eng = engine(256, 512, 1)
    cfg = eng.make_config(want_bounds=True)
    N = eng.points_per_frame(cfg)
    lengths = [1, 2, 31, 32, 33, 63, 64, 1023, 1024, 1025]
    vs = 0.01
    clouds = {f"runs lead={lead}": V.runs_cloud(lengths * 3, vs, rng, lead=lead) for lead in (0, 5, 31, 1000)}
    clouds["runs reversed"] = V.runs_cloud(lengths[::-1] * 3, vs, rng, lead=17)
    clouds["abab"] = V.abab_cloud(5000, vs, rng)
    clouds["scattered"] = V.scattered_cloud(60000, vs, rng)
    clouds["whole frame one voxel"] = V.one_voxel_cloud(N, rng, size=vs * 0.4, offset=(1.0, -2.0, 3.0))
    for name, p in clouds.items():
        _check(eng, cfg, [(p, V.colours(rng, len(p)))], vs, name)


def test_every_row_its_own_voxel_2m_rows(engine):
    """128^3 lattice, spacing 1, vs = 0.5: 2 097 152 voxels of one row each; the probe chains wrap at frame_cap and
    the 8-bit fingerprints collide."""
    rng = np.random.default_rng(7)
    eng = engine(1024, 2048, 1)
    cfg = eng.make_config(want_bounds=True)
    p = V.lattice_cloud(128, 1.0)
    assert len(p) == eng.points_per_frame(cfg) == 2097152
    got = _check(eng, cfg, [(p, V.colours(rng, len(p)))], 0.5, "lattice 128^3")
    assert len(got[0][0]) == len(p)


# ---- 4. packed-field limits --------------------------------------------------------------------
def test_one_voxel_of_16m_rows_and_the_row_limit(m, engine):
    """4095 x 4096 = 16 773 120 rows (the largest N below 2^24 at width 4096) in one voxel: with colours all 255 the
    packed sum r field reaches 4.277e9 of its 2^32 limit.  4096 x 4096 is refused (D2PC_ERR_UNSUPPORTED)."""
    import torch
    rng = np.random.default_rng(24)
    eng = engine(4095, 4096, 1)
    cfg = eng.make_config(want_bounds=True)
    N = eng.points_per_frame(cfg)
    assert N == 4095 * 4096 < (1 << 24)
    p = V.one_voxel_cloud(N, rng, size=10.0, offset=(-3.0, 1.0, 0.5))
    for kind in ("white", "black_white"):
        got = _check(eng, cfg, [(p, V.colours(rng, N, kind))], 100.0, f"16M rows {kind}")
        assert len(got[0][0]) == 1
    del p, got
    big = m.FrameEngine(4096, 4096, batch=1)
    cfg = big.make_config(want_bounds=True)
    z = torch.zeros((1, 4, 3), dtype=torch.float32, device=big.device)
    res = m.EmitResult(z, z.clone(), torch.zeros(1, dtype=torch.int32, device=big.device),
                       torch.zeros((1, 6), dtype=torch.float32, device=big.device))
    with pytest.raises(m.D2pcError) as e:
        big.voxel_downsample(cfg, res, 0.1)
    assert e.value.code == 4


# ---- 5. degenerate extents and voxels much larger than the cloud -------------------------------
@pytest.mark.parametrize("vs", [0.05, 1e3, 1e7, 1e9, 1e300])
def test_degenerate_extents_and_huge_voxels(engine, vs):
    """One point, three points, identical points, a plane, a line, an all-negative cloud, tight clusters (about 10
    units), as one batch.  The fixed point follows the cloud's extent, so a voxel of 1e9 or 1e300 keeps the means exact."""
    rng = np.random.default_rng(5)
    eng = engine(128, 128, 7)
    cfg = eng.make_config(want_bounds=True)
    clouds = V.degenerate_clouds(rng)
    frames = [(p, V.colours(rng, len(p))) for p in clouds.values()]
    got = _check(eng, cfg, frames, vs, f"degenerate vs={vs:g}")
    if vs >= 1e3:
        assert all(len(g[0]) == 1 for g in got)


# ---- 6. frames of different sizes sharing one table --------------------------------------------
def test_batch_of_different_frames_shares_one_table(engine):
    """Counts large, 0, 1, small, another large, all-one-voxel in one enqueue: every frame starts from the stale
    slots, flags and accumulators of the one before."""
    rng = np.random.default_rng(6)
    eng = engine(256, 512, 6)
    cfg = eng.make_config(want_bounds=True)
    N = eng.points_per_frame(cfg)
    vs = 0.02
    clouds = [_f(rng.random((N, 3)) * 3), np.zeros((0, 3), np.float32), _f([[0.5, 0.25, 2.0]]),
              _f(rng.random((100, 3))), V.runs_cloud([1, 33, 1025, 64] * 100, vs, rng, lead=9),
              V.one_voxel_cloud(50000, rng, size=vs * 0.3, offset=(4.0, 4.0, 4.0))]
    frames = [(p, V.colours(rng, len(p))) for p in clouds]
    got = _check(eng, cfg, frames, vs, "batch")
    want = [len(O.voxel_downsample(p, c, vs)[0]) for p, c in frames]
    assert [len(g[0]) for g in got] == want
    assert want[1] == 0 and want[2] == 1 and want[5] == 1
    # and the other way round: small frames first, the largest last
    _check(eng, cfg, frames[::-1], vs, "batch reversed")


def _f(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64).astype(np.float32))


# ---- 7. one engine, several configurations -----------------------------------------------------
def test_engine_reuses_its_table_across_densities(engine):
    """high -> medium -> low -> high -> medium on one engine, with and without z_range: the table is laid out for
    the config's rows per frame, so a new density must initialise it again."""
    rng = np.random.default_rng(8)
    eng = engine(240, 320, 2)
    for zr in (None, (0.5, 9.5)):
        for density in ("high", "medium", "low", "high", "medium"):
            cfg = eng.make_config(density=density, z_range=zr, want_bounds=True)
            N = eng.points_per_frame(cfg)
            frames = [(p, V.colours(rng, len(p))) for p in (_f(rng.random((N, 3)) * 2), _f(rng.random((N // 3, 3))))]
            _check(eng, cfg, frames, 0.05, f"{density} z_range={zr}")


def test_drop_in_api_across_densities(m):
    """The drop-in call caches one engine per geometry, not per density: a web request of another density must not
    fail (or return nothing) after the first."""
    H, W = 200, 300
    img = cases.make_image(H, W, 40)
    dep = cases.make_depth(H, W, 40, "scene")
    for zr in (None, (0.5, 9.5)):
        for density in ("high", "medium", "low", "high", "medium"):
            po, co = _oracle_rows(img, dep, density, zr)
            p, c, idx = m.depth_to_point_cloud(img, dep, density=density, z_range=zr, voxel_size=0.05,
                                               return_voxel_index=True)
            problems, _ = V.check_frame(p, c, idx, po, co, 0.05, f"drop-in {density} z_range={zr}")
            assert problems == [], problems


# ---- 8. the stage at densities medium and low -------------------------------------------------
@pytest.mark.parametrize("density,H,W", [("medium", 241, 323), ("low", 243, 329)])
def test_stage_voxels_at_medium_and_low(m, density, H, W):
    img = cases.make_image(H, W, 41)
    dep = cases.make_depth(H, W, 41, "scene")
    for zr in (None, (0.5, 9.5)):
        po, co = _oracle_rows(img, dep, density, zr)
        for vs in (0.05, 0.005, 0.5):
            p, c, idx = m.depth_to_point_cloud(img, dep, density=density, z_range=zr, voxel_size=vs,
                                               return_voxel_index=True)
            problems, _ = V.check_frame(p, c, idx, po, co, vs, f"stage {density} z_range={zr} vs={vs}")
            assert problems == [], problems


# ---- 9. input validation -----------------------------------------------------------------------
@pytest.mark.parametrize("vs", [0.0, -0.5, float("nan"), float("inf"), float("-inf")])
def test_voxel_size_must_be_finite_and_positive(m, vs):
    import torch
    eng = m.FrameEngine(16, 16, batch=1)
    cfg = eng.make_config(want_bounds=True)
    N = eng.points_per_frame(cfg)
    dev = eng.device
    res = m.EmitResult(torch.rand((1, N, 3), device=dev), torch.zeros((1, N, 3), device=dev),
                       torch.full((1,), N, dtype=torch.int32, device=dev), torch.zeros((1, 6), device=dev))
    with pytest.raises(ValueError):
        eng.voxel_downsample(cfg, res, vs)
    assert eng._voxel_table is None, "refused before any allocation or launch"
    img, dep = cases.make_image(16, 16, 1), cases.make_depth(16, 16, 1)
    with pytest.raises(ValueError):
        m.depth_to_point_cloud(img, dep, voxel_size=vs)


def test_fuzz_voxel_short():
    from profiles import fuzz_voxel
    assert fuzz_voxel.main(["fuzz_voxel", "40", "4716"]) == 0
