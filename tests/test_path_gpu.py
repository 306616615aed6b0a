"""GPU: the one-call path API (d2pc_path_enqueue) in all its modes equals the two-phase calls bit for bit,
the drop-in call is thread-safe, and engines work on a device that is not the current one."""
import threading
import warnings

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from tests import cases  # noqa: E402

pytestmark = pytest.mark.gpu


def _frames(B, H, W, h, w, seed):
    depth = np.stack([cases.make_depth(h, w, seed + i, "uniform") for i in range(B)])
    bgr = np.stack([cases.make_image(H, W, seed + i) for i in range(B)])
    return torch.from_numpy(depth).cuda(), torch.from_numpy(bgr).cuda()


@pytest.mark.parametrize("geom", [
    dict(H=216, W=384, h=216, w=384, B=9, kw={}),                               # native, ordered kernel eligible
    dict(H=216, W=384, h=130, w=231, B=7, kw={}),                               # resized (ring of materialised maps)
    dict(H=216, W=384, h=216, w=384, B=6, kw=dict(z_range=(0.5, 9.5))),        # masked
    dict(H=216, W=384, h=216, w=384, B=5, kw=dict(density="medium", want_bounds=True)),
    dict(H=33, W=47, h=20, w=31, B=4, kw={}),                                   # small frames (sort path), generic emit
])
def test_path_modes_equal_two_phase(geom):
    import image_to_pointcloud_b200 as m
    from image_to_pointcloud_b200 import _lib
    H, W, h, w, B, kw = (geom[k] for k in ("H", "W", "h", "w", "B", "kw"))
    depth, bgr = _frames(B, H, W, h, w, 300)
    eng = m.FrameEngine(H, W, h, w, batch=B, device="cuda:0")
    cfg = eng.make_config(**kw)
    s = torch.cuda.current_stream()
    n = eng.points_per_frame(cfg)

    def outputs():
        xyz, rgb = eng.alloc_outputs(cfg)
        xyz.fill_(-7.0); rgb.fill_(-7.0)
        cnt = torch.zeros(B, dtype=torch.int32, device="cuda")
        bounds = torch.zeros((B, 6), dtype=torch.float32, device="cuda") if cfg.want_bounds else None
        return xyz, rgb, cnt, bounds

    ref = outputs()
    eng.enqueue_stats(cfg, depth, s)
    eng.enqueue_status(cfg, s)
    eng.enqueue_emit(cfg, depth, bgr, ref[0], ref[1], ref[2], ref[3], s)
    torch.cuda.synchronize()
    assert int(eng._any_host[0]) == 0
    modes = [dict(), dict(graph=True), dict(sub_batch=2), dict(sub_batch=3, lookahead=2, graph=True),
             dict(sub_batch=2, flags=_lib.PATH_NO_OVERLAP), dict(flags=_lib.PATH_ORDERED, lookahead=3)]
    for mode in modes:
        for rep in range(2):   # twice: the cached graph is replayed the second time
            got = outputs() if rep == 0 else got
            eng.enqueue_path(cfg, depth, bgr, got[0], got[1], got[2], got[3], s, **mode)
            torch.cuda.synchronize()
            assert int(eng._any_host[0]) == 0, mode
            assert torch.equal(got[2], ref[2]), mode
            for b in range(B):
                k = int(ref[2][b])
                assert k <= n
                assert torch.equal(got[0][b, :k].view(torch.int32), ref[0][b, :k].view(torch.int32)), (mode, b)
                assert torch.equal(got[1][b, :k], ref[1][b, :k]), (mode, b)
            if cfg.want_bounds:
                assert torch.equal(got[3].view(torch.int32), ref[3].view(torch.int32)), mode


def test_path_flags_frames_for_fallback():
    """Frames the fast statistics decline (non-finite values) are flagged by the one-call path too, in every
    mode, and FrameEngine.process then finishes them through the exact fallback."""
    import image_to_pointcloud_b200 as m
    from image_to_pointcloud_b200 import _lib
    from oracle import d2pc_oracle as O
    H, W, B = 216, 384, 4
    depth = np.stack([cases.make_depth(H, W, 40 + i, "nonfinite" if i == 2 else "uniform") for i in range(B)])
    bgr = np.stack([cases.make_image(H, W, 40 + i) for i in range(B)])
    d_dev, b_dev = torch.from_numpy(depth).cuda(), torch.from_numpy(bgr).cuda()
    eng = m.FrameEngine(H, W, batch=B, device="cuda:0")
    cfg = eng.make_config()
    s = torch.cuda.current_stream()
    xyz, rgb = eng.alloc_outputs(cfg)
    cnt = torch.zeros(B, dtype=torch.int32, device="cuda")
    for mode in (dict(), dict(flags=_lib.PATH_ORDERED), dict(sub_batch=2)):
        eng.enqueue_path(cfg, d_dev, b_dev, xyz, rgb, cnt, None, s, **mode)
        torch.cuda.synchronize()
        assert int(eng._any_host[0]) == 1, mode
        assert eng._status.cpu().tolist() == [1, 1, 2, 1], mode
    res = eng.process(cfg, d_dev, b_dev)
    for b in range(B):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            po, co = O.depth_to_point_cloud(bgr[b], depth[b], density="high")
        assert np.array_equal(res.xyz[b].cpu().numpy().view(np.uint32), po.view(np.uint32)), b
        assert np.array_equal(res.rgb[b].cpu().numpy(), co), b


def test_drop_in_call_is_thread_safe():
    """Concurrent calls on ONE geometry (they share the cached engine and its staging buffers) must not mix
    their frames: each thread checks its own result against the oracle."""
    import image_to_pointcloud_b200 as m
    from oracle import d2pc_oracle as O
    H, W, h, w = 120, 160, 77, 103
    errors = []

    def worker(t):
        try:
            for i in range(6):
                img = cases.make_image(H, W, 1000 * t + i)
                dep = cases.make_depth(h, w, 1000 * t + i, "uniform")
                p, c = m.depth_to_point_cloud(img, dep, density="high", device="cuda:0", pinned=(i % 2 == 0))
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    po, co = O.depth_to_point_cloud(img, dep, density="high")
                if not (np.array_equal(p.view(np.uint32), po.view(np.uint32)) and np.array_equal(c, co)):
                    errors.append((t, i))
        except Exception as e:  # noqa: BLE001
            errors.append((t, repr(e)))

    threads = [threading.Thread(target=worker, args=(t,)) for t in range(4)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert errors == []


def test_stages_run_the_engine_under_its_lock(monkeypatch):
    """point_cloud_stage and depth_to_mesh share the cached engine with the drop-in call, so they run it under the
    same lock."""
    import image_to_pointcloud_b200 as m
    held = []
    process = m.FrameEngine.process

    def recording(self, *args, **kwargs):
        held.append(self._staging["lock"].locked())
        return process(self, *args, **kwargs)

    monkeypatch.setattr(m.FrameEngine, "process", recording)
    img, dep = cases.make_image(120, 160, 5), cases.make_depth(77, 103, 5, "uniform")
    m.point_cloud_stage(img, dep, output_format=None, device="cuda:0")
    m.depth_to_mesh(img, dep, device="cuda:0")
    assert held == [True, True]


def test_engine_on_a_device_that_is_not_current():
    """The library launches on the current device: FrameEngine makes its own device current around every call."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import image_to_pointcloud_b200 as m
    H, W, B = 64, 96, 2
    depth = np.stack([cases.make_depth(H, W, 5 + i, "uniform") for i in range(B)])
    bgr = np.stack([cases.make_image(H, W, 5 + i) for i in range(B)])
    outs = []
    for dev in ("cuda:0", "cuda:1"):
        torch.cuda.set_device(0)   # current device stays 0 while the engine lives on `dev`
        eng = m.FrameEngine(H, W, batch=B, device=dev)
        cfg = eng.make_config(z_range=(0.5, 9.5), want_bounds=True)
        res = eng.process(cfg, torch.from_numpy(depth).to(dev), torch.from_numpy(bgr).to(dev))
        vox = eng.voxel_downsample(cfg, res, 0.05)
        outs.append((res.xyz.cpu(), res.rgb.cpu(), res.count.cpu(), vox[3].cpu()))
    for a, b in zip(outs[0], outs[1]):
        assert torch.equal(a, b)


def test_stale_library_is_refused(monkeypatch, tmp_path):
    """A library built from other sources must not be loaded silently when the rebuild fails."""
    from image_to_pointcloud_b200 import _lib, build
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "build_library", lambda *a, **k: (_ for _ in ()).throw(RuntimeError("nvcc missing")))
    monkeypatch.setattr(build, "stored_digest", lambda: "0" * 64)
    with pytest.raises(RuntimeError, match="stale"):
        _lib.load_library()


@pytest.mark.parametrize("density", ["medium", "low"])
@pytest.mark.parametrize("kind", ["uniform", "scene", "ties"])
def test_masked_strided_fast_path(density, kind):
    """density medium / low with a depth-range mask (what the reference UI's default density gives with the
    extension on) runs the vectorised masked emit: rows, order and count equal the oracle's post-filter."""
    import image_to_pointcloud_b200 as m
    from oracle import d2pc_oracle as O
    H, W = 150, 224     # W % 16 == 0: the fast path for both strides; H not a multiple of the stride
    for h, w in ((H, W), (97, 131)):
        img = cases.make_image(H, W, 77)
        dep = cases.make_depth(h, w, 78, kind)
        for zr in ((0.5, 9.5), (9.0, 9.99), (0.0, 0.2)):
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                po, co = O.depth_to_point_cloud(img, dep, density=density)
            keep = O.range_mask(po, *zr)
            p, c = m.depth_to_point_cloud(img, dep, density=density, z_range=zr, device="cuda:0")
            assert p.shape[0] == int(keep.sum()), (h, w, zr)
            assert np.array_equal(p.view(np.uint32), po[keep].view(np.uint32)), (h, w, zr)
            assert np.array_equal(c, co[keep]), (h, w, zr)
