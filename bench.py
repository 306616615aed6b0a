#!/usr/bin/env python
"""bench.py -- throughput of the depth-map -> coloured point-cloud stage on B200.

    python bench.py --gpus N --steps K --warmup W            (ours; torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...  (CPU arm, rank 0 only)
    python bench.py ... --dump-outputs DIR                   (also save what the last timed step returned)

A *step* is one pass of the whole hot path (exact percentile statistics + fused emit, one library
call: d2pc_path_enqueue, replayed as a CUDA graph) over one batch of synthetic frames.  Workload at every N: BASELINE.json configs[1] -- 1920x1080 frames,
native-size float32 depth + uint8 BGR, density "high" (stride 1), invert, depth_scale 10, every
point kept (the reference has no mask) -- ``--batch`` frames per GPU per step (weak scaling:
frames are independent, sharded by frame, no collective on the data path).

value   Mpoints/s, whole job, inputs resident in HBM, CUDA-event timed, max over ranks.
e2e     same metric through the host API (HostFramePipeline.run_pinned): pinned HOST buffers in,
        pinned HOST buffers out, H2D and D2H inside the timed region.
roofline  the dominant kernel (emit): algorithmic bytes (4 B depth + 3 B BGR + 24 B out per
        point, SURVEY.md 8d) / its CUDA-event duration, against MEASURED_PEAKS.json hbm_gbs.
cpu_baseline  the UNMODIFIED reference function (baseline/_ref/backend/app.py, copied from
        /root/reference by __graft_entry__.build(); the oracle's loop-faithful port if that copy is
        absent) timed on one host core on a bounded sample (rank 0, N = 1 only).
extras  (N = 1) the other BASELINE.json configurations, device-resident: 1080p with a DA-v2-sized
        depth map, 4K native, configs[2] (4K + z-range + 5 mm voxels), configs[4] (voxel sweep).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "depth_to_point_cloud_throughput"
UNIT = "Mpoints/s"
IMG_H, IMG_W = 1080, 1920
BYTES_PER_POINT_ALG = 4 + 3 + 24  # SURVEY.md 8d: native depth, stride 1, no mask
FALLBACK_HBM_GBS = 6650.0         # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--batch", type=int, default=128, help="frames per GPU per step")
    ap.add_argument("--e2e-frames", type=int, default=32, help="frames per e2e step (0: same as --batch)")
    ap.add_argument("--chunk", type=int, default=8, help="frames per pipeline chunk in the e2e path")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the other BASELINE configurations (N = 1)")
    ap.add_argument("--extras-full", action="store_true", help="also writers / outlier removal / single-call latency")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (a fixed sample of the rows)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs saves the GPU path's outputs; the reference arm has none")
    return args


def config_dict(args, n_gpus):
    return {
        "workload": "configs[1]: 1920x1080 frames, native-size f32 depth + u8 BGR, density=high, invert, "
                    "depth_scale=10, all points kept",
        "frames_per_gpu_per_step": args.batch,
        "points_per_frame": IMG_H * IMG_W,
        "global_frames_per_step": args.batch * n_gpus,
        "parallelism": f"frame-sharded x{n_gpus}, no collective",
        "l2_hygiene": "per-step inputs (%.0f MB) and outputs (%.0f MB) per GPU exceed the 126 MB L2"
                      % (args.batch * IMG_H * IMG_W * 7 / 1e6, args.batch * IMG_H * IMG_W * 24 / 1e6),
    }


# ----------------------------------------------------------------------------------------------
# clocks sampler (NVML), runs during the timed region
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
            "hw_power_brake": getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80),
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.005)

    def __enter__(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr is not None:
            self._thr.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def measured_traffic_per_frame():
    """dram__bytes_read.sum + dram__bytes_write.sum of emit_fast_kernel per 1080p frame, from the
    committed `ncu --set full` capture (profiles/r02_emit_traffic.json); None if absent."""
    try:
        ps = [os.path.join(ROOT, "profiles", r + "_emit_traffic.json") for r in ("r02", "r01")]
        p = [x for x in ps if os.path.exists(x)][0]
        d = json.load(open(p))
        return float(d["dram_bytes_per_frame"])
    except Exception:
        return None


def pcie_ceiling(n_gpus):
    """End-to-end ceiling of this pool's boxes in Mpoints/s for n_gpus GPUs copying concurrently: plain pinned
    cudaMemcpyAsync in both directions at the pipeline's sizes (profiles/pcie_ceiling.py -> r02_pcie_ceiling.json)."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r02_pcie_ceiling.json")))
        for r in d["runs"]:
            if r["gpus"] == n_gpus and r["mode"] == "both":
                return r
    except Exception:
        pass
    return None


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


# ----------------------------------------------------------------------------------------------
# synthetic frames (SURVEY.md 8d C2/C4: frame i seeded 1000 + i)
# ----------------------------------------------------------------------------------------------
def synth_frames_device(n, device, seed0):
    """Device-side generation of n synthetic frames (uniform*20 depth, random BGR).  Statistically
    the same as tests/cases.py; generated on the GPU because 1024 host-generated 1080p frames
    would take minutes."""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed0)
    depth = torch.rand((n, IMG_H, IMG_W), generator=g, device=device, dtype=torch.float32) * 20.0
    bgr = torch.randint(0, 256, (n, IMG_H, IMG_W, 3), generator=g, device=device, dtype=torch.uint8)
    return depth, bgr


DUMP_SAMPLE_POINTS = 1 << 20  # 24 MB of xyz + rgb rows; a whole step's output is 24 B per point


def dump_outputs(out_dir, xyz, rgb, count, prefix=""):
    """Save what the path returned: the per-frame point counts, and the xyz and rgb rows at a fixed sample of
    (frame, point) positions, drawn with seed 0 and sorted, so that two builds can be compared file for file."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    total = xyz.shape[0] * xyz.shape[1]
    idx = np.sort(np.random.default_rng(0).choice(total, min(DUMP_SAMPLE_POINTS, total), replace=False))
    sel = torch.from_numpy(idx).to(xyz.device)
    arrays = {"count": count.cpu().numpy().astype(np.float64),
              "xyz_sample": xyz.reshape(-1, 3)[sel].cpu().numpy(),
              "rgb_sample": rgb.reshape(-1, 3)[sel].cpu().numpy()}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), a)


# ----------------------------------------------------------------------------------------------
# CPU arm
# ----------------------------------------------------------------------------------------------
_REF_FN = None       # set in the parent before the worker pool forks
_REF_KIND = "port"


def _load_cpu_reference():
    """The stock reference function when its copy travelled with the repo, else the oracle's port."""
    global _REF_FN, _REF_KIND
    if _REF_FN is not None:
        return _REF_FN, _REF_KIND
    try:
        from baseline import ref_arm
        if ref_arm.available():
            _REF_FN, _REF_KIND = ref_arm.load(), "reference"
            return _REF_FN, _REF_KIND
    except Exception as e:  # missing dependency of app.py on this box: say so, use the port
        print("reference copy not loadable (%s): using the oracle's port" % e, file=sys.stderr)
    from oracle import d2pc_oracle as O
    _REF_FN, _REF_KIND = O.depth_to_point_cloud_loop, "port"
    return _REF_FN, _REF_KIND


def _cpu_loop_job(job):
    """One bounded sample: the reference function on an (h x w) native-depth frame."""
    h, w, seed = job
    from tests import cases
    fn, _ = _load_cpu_reference()
    img = cases.make_image(h, w, seed)
    dep = cases.make_depth(h, w, seed, "uniform")
    t0 = time.perf_counter()
    p, c = fn(img, dep, density="high")
    return len(p), time.perf_counter() - t0


def cpu_baseline_single_core():
    """Rank 0, N = 1: one core, a quarter-height 1080p frame (270 x 1920 = 518 400 points, ~1.5 s); the
    per-point cost of the reference's Python loop does not depend on the frame size."""
    from oracle import d2pc_oracle as O
    from tests import cases
    fn, kind = _load_cpu_reference()
    h, w = 270, 1920
    n, dt = _cpu_loop_job((h, w, 1))
    img = cases.make_image(IMG_H, IMG_W, 1)
    dep = cases.make_depth(IMG_H, IMG_W, 1, "uniform")
    t0 = time.perf_counter()
    O.depth_to_point_cloud(img, dep, density="high")
    dv = time.perf_counter() - t0
    what = ("the unmodified reference depth_to_point_cloud (baseline/_ref/backend/app.py:174-250)" if kind == "reference"
            else "oracle.depth_to_point_cloud_loop (line-for-line port of app.py:183-246)")
    return {"value": round(n / dt / 1e6, 4), "unit": UNIT, "cores": 1, "kind": kind,
            "cores_available": os.cpu_count(),
            "sample": "%s on one 270x1920 native-depth frame, density=high (%d points, %.2f s)" % (what, n, dt),
            "vectorised_numpy_port_mpoints_s": round(IMG_H * IMG_W / dv / 1e6, 3)}


def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path -- the unmodified
    backend/app.py::depth_to_point_cloud from baseline/_ref (the oracle's port only if that copy is missing) --
    on every host core: one forked process per core, each step one bounded sample per core (a 135 x 1920
    native-depth frame = 1/8 of a 1080p frame; the per-point cost of the Python loop does not depend on the
    frame size)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    fn, kind = _load_cpu_reference()   # imported once here; the workers are forked from this process
    cores = os.cpu_count() or 1
    h, w = 135, 1920
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        jobs = lambda s: [(h, w, 1000 + s * cores + i) for i in range(cores)]  # noqa: E731
        for s in range(args.warmup):
            pool.map(_cpu_loop_job, jobs(s))
        t0 = time.perf_counter()
        pts = 0
        for s in range(args.steps):
            pts += sum(n for n, _ in pool.map(_cpu_loop_job, jobs(args.warmup + s)))
        dt = time.perf_counter() - t0
    val = pts / dt / 1e6
    cfg = config_dict(args, args.gpus)
    # what this arm really processed per step: a bounded sample of the same workload (same frame content, knobs
    # and per-point work), sized for the CPU -- not the GPU arm's 128 frames per step
    eq = round(cores * h * w / (IMG_H * IMG_W), 3)
    cfg["frames_per_gpu_per_step"] = eq
    cfg["global_frames_per_step"] = eq
    cfg["parallelism"] = "%d host processes, one bounded sample each per step" % cores
    cfg.pop("l2_hygiene", None)
    cfg["reference_arm_step"] = {"frames": cores, "frame_shape": [h, w], "points": cores * h * w,
                                 "equivalent_1080p_frames": round(cores * h * w / (IMG_H * IMG_W), 3),
                                 "processes": cores, "implementation": kind}
    what = ("unmodified reference backend/app.py::depth_to_point_cloud" if kind == "reference"
            else "oracle.depth_to_point_cloud_loop (port)")
    line = {
        "impl": "reference", "metric": METRIC, "value": round(val, 4), "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt / args.steps * 1e3, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": cfg,
        "images_per_s": round(val * 1e6 / (IMG_H * IMG_W), 4),
        "cpu_baseline": {"value": round(val, 4), "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": "per step and core: %s on one 135x1920 native-depth frame (1/8 of a 1080p "
                                   "frame), density=high" % what},
        "e2e": {"value": round(val, 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun --nproc-per-node %d for --gpus %d" % (args.gpus, args.gpus))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    # pin this rank to the CPUs next to its GPU before any pinned buffer is allocated (the e2e leg streams
    # ~65 MB per frame through host memory; a remote NUMA node halves that)
    try:
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local_rank))
    except Exception:
        pass
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    import image_to_pointcloud_b200 as m
    from image_to_pointcloud_b200 import shard_frames

    B, K, Wu = args.batch, args.steps, args.warmup
    # frame-sharded: rank r owns global frames shard_frames(B*world, world, r)
    my_frames = shard_frames(B * world, world, rank)
    assert len(my_frames) == B
    depth, bgr = synth_frames_device(B, device, 1000 + my_frames.start)
    eng = m.FrameEngine(IMG_H, IMG_W, batch=B, img_c=3, device=device)
    cfg = eng.make_config(density="high", invert=True, depth_scale=10.0)
    xyz, rgb = eng.alloc_outputs(cfg)
    count = torch.zeros(B, dtype=torch.int32, device=device)
    stream = torch.cuda.current_stream(device)
    n_points = eng.points_per_frame(cfg)

    def step():
        # statistics + status + emit in one library call, replayed as a CUDA graph
        eng.enqueue_path(cfg, depth, bgr, xyz, rgb, count, None, stream, graph=True)
    launches_per_step = 3 + 1 + 1  # sample, scan, select | emit | status

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    for _ in range(Wu):
        step()
    barrier()
    # correctness of what is being timed: every frame finished on the fast path and frame 0 matches
    assert int(eng._any_host[0]) == 0, "a synthetic frame needed the fallback path"
    assert int(count.min()) == n_points and int(count.max()) == n_points

    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        barrier()
        ev0.record(stream)
        for _ in range(K):
            step()
        ev1.record(stream)
        barrier()
    ms_total = ev0.elapsed_time(ev1)
    assert int(eng._any_host[0]) == 0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, xyz, rgb, count, "" if world == 1 else "rank%d_" % rank)
    if rank == 0:
        # what was timed is checked against the oracle: one frame of the timed output, bit for bit
        import warnings

        import numpy as np
        from oracle import d2pc_oracle as O  # checker only
        fchk = B // 2
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            po, co = O.depth_to_point_cloud(bgr[fchk].cpu().numpy(), depth[fchk].cpu().numpy(), density="high")
        got_p, got_c = xyz[fchk].cpu().numpy(), rgb[fchk].cpu().numpy()
        assert np.array_equal(got_p.view(np.uint32), po.view(np.uint32)), "timed frame: xyz differs from the oracle"
        assert np.array_equal(got_c, co), "timed frame: rgb differs from the oracle"

    # dominant kernel alone (emit), CUDA events on the same stream, same buffers (> L2)
    emit_iters = K
    for _ in range(3):
        eng.enqueue_emit(cfg, depth, bgr, xyz, rgb, count, None, stream)
    torch.cuda.synchronize(device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(emit_iters):
        eng.enqueue_emit(cfg, depth, bgr, xyz, rgb, count, None, stream)
    e1.record(stream)
    torch.cuda.synchronize(device)
    emit_ms = e0.elapsed_time(e1) / emit_iters
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record(stream)
    for _ in range(emit_iters):
        eng.enqueue_stats(cfg, depth, stream)
    s1.record(stream)
    torch.cuda.synchronize(device)
    stats_ms = s0.elapsed_time(s1) / emit_iters

    # end to end through the host API: pinned host in -> pinned host out
    ef = args.e2e_frames or B
    pipe = m.HostFramePipeline(IMG_H, IMG_W, img_c=3, chunk=min(args.chunk, ef), density="high", device=device)
    h_img, h_dep = pipe.alloc_pinned_inputs(ef)
    sel = torch.arange(ef, device=device) % B  # e2e frames = the device-resident frames (repeated if ef > B)
    h_dep.copy_(depth[sel].cpu())
    h_img.copy_(bgr[sel].cpu())
    o_xyz, o_rgb, o_cnt = pipe.alloc_pinned_outputs(ef)
    e2e_steps = K
    for _ in range(2):
        pipe.run_pinned(h_img, h_dep, o_xyz, o_rgb, o_cnt)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        pipe.run_pinned(h_img, h_dep, o_xyz, o_rgb, o_cnt)
    torch.cuda.synchronize(device)
    e2e_s = time.perf_counter() - t0
    # the e2e result is the same bits as the device-resident result
    assert torch.equal(o_xyz[0], xyz[0].cpu()) and int(o_cnt[0]) == n_points
    h2d_f, d2h_f = pipe.bytes_per_frame()

    # max over ranks
    t = torch.tensor([ms_total, e2e_s, emit_ms, stats_ms], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, e2e_s, emit_ms, stats_ms = (float(x) for x in t.cpu())

    extras = {}
    if world == 1 and rank == 0 and not args.no_extras:
        extras = run_extras(m, device, full=args.extras_full)

    if rank == 0:
        peak, peak_src = measured_peak()
        pts_step = B * world * n_points
        value = pts_step * K / (ms_total * 1e-3) / 1e6
        emit_bytes = B * n_points * BYTES_PER_POINT_ALG
        achieved = emit_bytes / (emit_ms * 1e-3) / 1e9
        path_gbs = B * n_points * BYTES_PER_POINT_ALG * K / (ms_total * 1e-3) / 1e9
        e2e_val = ef * world * n_points * e2e_steps / e2e_s / 1e6
        line = {
            "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wu,
            "ms_per_step": round(ms_total / K, 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_dict(args, world),
            "images_per_s": round(value * 1e6 / n_points, 1),
            "e2e": {"value": round(e2e_val, 2), "unit": UNIT, "h2d_bytes_per_step": h2d_f * ef,
                    "d2h_bytes_per_step": d2h_f * ef, "frames_per_step": ef, "steps": e2e_steps,
                    "images_per_s": round(e2e_val * 1e6 / n_points, 1),
                    "api": "HostFramePipeline.run_pinned (pinned host in/out, 3 streams, chunk=%d)" % pipe.chunk},
            "gpu_launches": launches_per_step * K,
            "oracle_check": "frame %d of the timed output equals oracle.depth_to_point_cloud bit for bit" % (B // 2),
            "roofline": {"bound": "hbm", "kernel": "emit_fast_kernel", "achieved": round(achieved, 1),
                         "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                         "traffic": (round(measured_traffic_per_frame() * B) if measured_traffic_per_frame() else None),
                         "peak_source": peak_src, "alg_bytes_per_launch": emit_bytes,
                         "launch_ms": round(emit_ms, 4),
                         "whole_path_gbs_per_gpu": round(path_gbs, 1),
                         "whole_path_frac": round(path_gbs / peak, 4),
                         "stats_ms_per_step": round(stats_ms, 4)},
            "clocks": clocks.summary(),
        }
        ceil = pcie_ceiling(world)
        if ceil and ceil.get("e2e_ceiling_mpoints_s"):
            line["e2e"]["pcie_ceiling_mpoints_s"] = ceil["e2e_ceiling_mpoints_s"]
            line["e2e"]["frac_of_pcie_ceiling"] = round(e2e_val / ceil["e2e_ceiling_mpoints_s"], 3)
            line["e2e"]["pcie_ceiling_source"] = ("profiles/r02_pcie_ceiling.json: %d GPU(s) copying concurrently, plain pinned "
                                                  "cudaMemcpyAsync both ways: %.1f GB/s D2H + %.1f GB/s H2D aggregate"
                                                  % (world, ceil["d2h_gbs_aggregate"], ceil["h2d_gbs_aggregate"]))
        if extras:
            line["extras"] = extras
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_single_core()
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_extras(m, device, full=False):
    """The other BASELINE.json configurations, device-resident, CUDA-event timed (not the headline).  Every
    entry carries its algorithmic bytes (SURVEY.md 8d: 4 D + 3 N + 24 N_out per frame), ms and the fraction of
    the measured copy bandwidth."""
    import torch
    out = {}
    peak = measured_peak()[0]

    def timeit(fn, iters=10):
        for _ in range(3):
            fn()
        torch.cuda.synchronize(device)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        torch.cuda.synchronize(device)
        return a.elapsed_time(b) / iters

    g = torch.Generator(device=device)
    g.manual_seed(5)
    variants = {
        "1080p_dav2_depth_518x924 (every real request resizes, app.py:186-188)": (1080, 1920, 518, 924, 64, None, "high"),
        "1080p_dav2_depth_density_medium (what the reference UI runs)": (1080, 1920, 518, 924, 64, None, "medium"),
        "1080p_native_zrange_0.5_9.5": (1080, 1920, 1080, 1920, 64, (0.5, 9.5), "high"),
        "1080p_native_zrange_density_medium": (1080, 1920, 1080, 1920, 64, (0.5, 9.5), "medium"),
        "4k_native": (2160, 3840, 2160, 3840, 16, None, "high"),
        "4k_native_zrange_0.5_9.5": (2160, 3840, 2160, 3840, 16, (0.5, 9.5), "high"),
    }
    for name, (H, W, h, w, B, zr, dens) in variants.items():
        eng = m.FrameEngine(H, W, h, w, batch=B, device=device)
        cfg = eng.make_config(density=dens, z_range=zr)
        depth = torch.rand((B, h, w), generator=g, device=device) * 20
        bgr = torch.randint(0, 256, (B, H, W, 3), generator=g, device=device, dtype=torch.uint8)
        xyz, rgb = eng.alloc_outputs(cfg)
        cnt = torch.zeros(B, dtype=torch.int32, device=device)
        s = torch.cuda.current_stream(device)

        def step():
            eng.enqueue_path(cfg, depth, bgr, xyz, rgb, cnt, None, s, graph=True)
        ms = timeit(step)
        kept = int(cnt.sum())
        n_frame = eng.points_per_frame(cfg)
        alg = B * (4 * h * w + 3 * n_frame) + 24 * kept   # SURVEY 8d: 4 D + 3 N + 24 N_out per frame
        out[name] = {"ms_per_step": round(ms, 4), "frames": B, "mpoints_out_per_s": round(kept / ms / 1e3, 1),
                     "images_per_s": round(B / ms * 1e3, 1), "kept_fraction": round(kept / (B * n_frame), 4),
                     "alg_bytes": alg, "alg_gbs": round(alg / ms / 1e6, 1), "frac_of_measured_peak": round(alg / ms / 1e6 / peak, 4)}
        del eng, depth, bgr, xyz, rgb
        torch.cuda.empty_cache()
    # BASELINE configs[2] / [4]: 4K frame, depth-range mask, voxel-size sweep (voxel stage alone)
    from profiles.voxel_sweep import sweep
    sw = sweep(iters=5, peak=peak)
    out["configs[4] 4k_zrange_voxel_sweep (voxel stage alone)"] = sw
    # configs[2]: one 4K frame through statistics + masked emit + 5 mm voxel grid (smooth scene)
    from profiles.voxel_sweep import config2
    out["configs[2] 4k_zrange_voxel_5mm (whole call)"] = config2(peak=peak)
    if full:
        # row f3: writer byte layouts on one 1080p cloud (kernels only)
        from profiles.writers_bench import bench as writers_bench
        out["writers_1080p"] = writers_bench()
        # row f1: statistical outlier removal on the stage's own clouds
        from profiles.sor_bench import bench as sor_bench
        out["sor_k20"] = sor_bench()
        # the drop-in call itself: NumPy in, NumPy out, one image (what backend/app.py:468 does per request)
        import numpy as np
        rng = np.random.default_rng(1)
        lat = {}
        for name, (H, W, h, w, dens) in {"480p_dav2_medium (UI default)": (480, 640, 518, 686, "medium"),
                                         "1080p_dav2_high": (1080, 1920, 518, 924, "high"),
                                         "1080p_native_high": (1080, 1920, 1080, 1920, "high"),
                                         "4k_dav2_high": (2160, 3840, 518, 924, "high")}.items():
            img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
            dep = (rng.random((h, w)) * 20).astype(np.float32)
            for _ in range(3):
                p, c = m.depth_to_point_cloud(img, dep, density=dens, device=device)
            ts = []
            for _ in range(10):
                t0 = time.perf_counter()
                p, c = m.depth_to_point_cloud(img, dep, density=dens, device=device)
                ts.append(time.perf_counter() - t0)
            ts.sort()
            lat[name] = {"points": len(p), "median_ms": round(ts[5] * 1e3, 3), "mpoints_per_s": round(len(p) / ts[5] / 1e6, 1)}
        out["single_call_latency_numpy_in_out"] = lat
    return out


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
