#!/usr/bin/env python
"""Benchmark of the Tracker hot path on B200 (BASELINE.json metric: particle-updates/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]

Workload (``config.workload``): BASELINE.json configs[1] — single nadir observer, CartesianMotion,
1 000 points x 10 000 particles x 100 frames, full k1-k6/p1/p2 distortion, 15x15 template, synthetic
translated-texture 4288x2848 uint8 frames.  One "step" = one whole ``track`` of that workload.

* ``value``   device-resident inputs (frames already in HBM), CUDA-event time around ``gb_track`` (every update
              of every point, batches of points advancing on their own streams) plus — for N > 1 — the final
              NCCL all-gather of the results.  Points x particles x frames of ALL ranks / max-over-ranks time.
              Weak scaling: every rank tracks its own 1 000 points.
* ``e2e``     the same metric through the public ``Tracker.track`` call with the frames in pinned HOST
              memory: per step the H2D copy of all frames + model tables and the D2H read of means /
              sigmas / status are inside the timed region.
* ``roofline`` for the dominant kernel ``k_s4p_resample_propagate``: algorithmic bytes per launch (96 B x the
              particles of a launch, SURVEY.md §8d) / its mean duration from CUDA events recorded around every
              launch on the launching stream (``gb_kernel_timing``; one untimed extra track with all points in
              one batch so that launches do not overlap), against MEASURED_PEAKS.json ``hbm_gbs``.
              ``whole_update`` is the same figure for a complete update (all kernels) inside the timed region;
              ``kernels`` / ``kernels_serial`` list every kernel's time per track in the production plan
              (overlapping streams) and alone.
* ``cpu_baseline`` the NumPy/SciPy/OpenCV oracle (a port of the Python reference, ``oracle/``) timed on one
              host core on a bounded sub-sample of the same workload (full N, fewer points and frames).
* ``--impl reference`` times that CPU port with every host core (fork pool over points, the reference's
              own parallel axis) and prints the same JSON line with ``"impl": "reference"``.
* ``--dump-outputs DIR`` writes what the last timed ``gb_track`` computed (``dump_outputs``), so that two builds can be
              compared output for output: the inputs are seeded, the same arguments give the same inputs.
"""
import argparse
import datetime
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "particle_updates_per_s"
UNIT = "particle-updates/s"
# DRAM bytes per particle of k_s4p_resample_propagate from the ncu --set full capture (profiles/r1_summary.md)
S4P_DRAM_BYTES_PER_PARTICLE = 99.0
ALGORITHMIC_BYTES_PER_UPDATE = 96.0  # read 6 x f64 parent state + write 6 x f64 child state (SURVEY.md §8d)

# BASELINE.json configs that fit one GPU.  `scene`: keyword arguments of synthetic.nadir_scene (n_points = points per GPU),
# `second`: add the second station (rolled by 180 deg, one frame later: staggered templates), `bytes`: algorithmic HBM bytes per
# particle-update (SURVEY.md §8d: read + write of the 6 x f64 state; + 24 B where the elevation likelihood reads x, y, z again),
# `cpu`: (points, frames) of the bounded CPU sample.
CONFIGS = {
    1: dict(name="configs[0]: 1 observer, CartesianMotion, 10 points x 1000 particles x 20 frames, 15x15 template, 600x400 uint8 frames",
            scene=dict(n_points=10, n_particles=1000, n_frames=20, imgsz=(600, 400), seed=1), second=False, bytes=96.0, cpu=(10, 20)),
    2: dict(name="configs[1]: 1 observer, CartesianMotion, 1000 points x 10000 particles x 100 frames, "
                 "full k1-k6/p1/p2, 15x15 template, 4288x2848 uint8 frames",
            scene=dict(n_points=1000, n_particles=10000, n_frames=100, imgsz=(4288, 2848), velocity_sigma=0.2, seed=2, margin_px=200),
            second=False, bytes=96.0, cpu=(40, 50)),
    3: dict(name="configs[2]: CylindricalMotion (dem_sigma = 1 m), 2 observers, 10000 points x 10000 particles x 100 frames, 4288x2848",
            scene=dict(n_points=10000, n_particles=10000, n_frames=100, imgsz=(4288, 2848), kind="cylindrical", velocity_sigma=0.2,
                       seed=3, margin_px=200), second=True, bytes=120.0, cpu=(8, 10)),
    4: dict(name="configs[3]: 31x31 template / ~100 px search windows, 1000 points x 100000 particles x 50 frames, 4288x2848",
            scene=dict(n_points=1000, n_particles=100000, n_frames=50, imgsz=(4288, 2848), tile_size=(31, 31), velocity_sigma=0.3,
                       seed=4, margin_px=300), second=False, bytes=96.0, cpu=(4, 10)),
}
WORKLOAD = dict(CONFIGS[2]["scene"])
WORKLOAD_NAME = CONFIGS[2]["name"]
ACTIVE = {"config": 2}


def select_config(number):
    """Make BASELINE.json config `number` the workload of this process (bench.py --config)."""
    global WORKLOAD, WORKLOAD_NAME, ALGORITHMIC_BYTES_PER_UPDATE
    ACTIVE["config"] = number
    WORKLOAD = dict(CONFIGS[number]["scene"])
    WORKLOAD_NAME = CONFIGS[number]["name"]
    ALGORITHMIC_BYTES_PER_UPDATE = CONFIGS[number]["bytes"]


def second_station(scene):
    """Same place, rolled 180 deg (frames flipped both ways), radial-only distortion, first image one frame later."""
    from glimpse_b200 import synthetic

    first = scene.observers[0]
    frames, cams, dts = [], [], []
    for t in range(1, len(first.frames)):
        frames.append(np.ascontiguousarray(first.frames[t][::-1, ::-1]))
        vec = first.cams[t].copy()
        vec[3:6] = (0.0, -90.0, 180.0)
        vec[18:20] = 0.0
        cams.append(vec)
        dts.append(first.datetimes[t])
    scene.observers.append(synthetic.ObserverScene(frames, np.array(cams), dts, sigma=0.4))
    return scene


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons of one GPU sampled every ~10 ms during the timed region, through NVML
    (``pynvml``) in a thread; falls back to polling ``nvidia-smi`` when NVML cannot be loaded."""

    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = self.path = self.thread = None
        self.sm, self.smax, self.reasons = [], [], set()

    def _nvml_loop(self, nv, handle):
        names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(handle, nv.NVML_CLOCK_SM)))
                self.smax.append(float(nv.nvmlDeviceGetMaxClockInfo(handle, nv.NVML_CLOCK_SM)))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(handle)
                for name, bit in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.01)

    def start(self):
        try:
            import threading

            import pynvml as nv

            nv.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            index = int(visible.split(",")[self.index]) if visible and visible.split(",")[self.index].isdigit() else self.index
            handle = nv.nvmlDeviceGetHandleByIndex(index)
            self._stop = threading.Event()
            self.thread = threading.Thread(target=self._nvml_loop, args=(nv, handle), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.QUERY}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.thread is not None:
            self._stop.set()
            self.thread.join(timeout=2)
        elif self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
            for line in open(self.path):
                parts = [p.strip() for p in line.split(",")]
                if len(parts) < 9:
                    continue
                try:
                    self.sm.append(float(parts[1]))
                    self.smax.append(float(parts[2]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                    if val.lower().startswith("active"):
                        self.reasons.add(name)
            os.unlink(self.path)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": float(max(self.smax)), "reasons": sorted(self.reasons),
                "samples": len(self.sm)}


def dump_outputs(directory, result, limit=64 * 10 ** 6):
    """Write the arrays ``Session.fetch`` returns (means, sigmas, status, status_time, obs_flags) as ``directory/<name>.npy``,
    float64 (obs_flags: float32, exact for its uint8 values), and the point each row belongs to as ``points.npy``.  When all
    points would take more than ``limit`` bytes, a fixed seeded sample of the points is written."""
    arrays = {k: np.asarray(result[k], dtype=np.float32 if k == "obs_flags" else np.float64)
              for k in ("means", "sigmas", "status", "status_time", "obs_flags")}
    P = len(arrays["means"])
    per_point = 8 + sum(a[0].nbytes for a in arrays.values())
    budget = limit - 1024 * (len(arrays) + 1)  # (.npy headers)
    points = np.arange(P)
    if P * per_point > budget:
        points = np.sort(np.random.default_rng(0).choice(P, budget // per_point, replace=False))
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "points.npy"), points.astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), np.ascontiguousarray(a[points]))


def build_scene(n_points, n_frames, pinned=False):
    from glimpse_b200 import synthetic

    kw = dict(WORKLOAD)
    kw.update(n_points=n_points, n_frames=n_frames)
    scene = synthetic.nadir_scene(**kw)
    if CONFIGS[ACTIVE["config"]]["second"]:
        scene = second_station(scene)
    if pinned:
        import torch

        for obs in scene.observers:
            frames = []
            for f in obs.frames:
                t = torch.empty(f.shape, dtype=torch.uint8).pin_memory()
                t.numpy()[...] = f
                frames.append(t.numpy())
            obs.frames = frames
    return scene


# --------------------------------------------------------------------------------------------------
# CPU legs (oracle = NumPy/SciPy/OpenCV port of the Python reference)
# --------------------------------------------------------------------------------------------------
_SCENE = None  # inherited by forked workers (frames are not pickled)


def _cpu_track_block(args):
    import warnings

    import helpers
    from oracle import tracker_oracle as orc

    lo, hi, seed = args
    scene = _SCENE
    try:
        import cv2

        cv2.setNumThreads(1)
    except Exception:
        pass
    obs, models, taus, index = helpers.oracle_inputs(scene, points=range(lo, hi))
    np.random.seed(seed + lo)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        res = orc.track(obs, models, taus, index, tile_size=scene.tile_size, raise_errors=False)
    return int(np.isfinite(res.means[:, -1, 0]).sum())


def cpu_rate(scene, n_points, cores):
    """particle-updates/s of the CPU port on `cores` processes (points split into contiguous blocks)."""
    global _SCENE
    _SCENE = scene
    T = len(scene.observers[0].frames)
    t0 = time.perf_counter()
    if cores == 1:
        _cpu_track_block((0, n_points, 11))
    else:
        import multiprocessing as mp

        per = -(-n_points // cores)
        blocks = [(lo, min(lo + per, n_points), 11) for lo in range(0, n_points, per)]
        with mp.get_context("fork").Pool(cores) as pool:
            pool.map(_cpu_track_block, blocks)
    dt = time.perf_counter() - t0
    return n_points * scene.n_particles * T / dt, dt


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    cores = max(1, len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    cores = min(cores, 64)
    cfg = CONFIGS[ACTIVE["config"]]
    # config 2: 4 points per core x half of the workload's frames (search windows grow with time, so do the costs); the
    # other configs: their bounded CPU sample per core group
    n_points, n_frames = (4 * cores, 50) if ACTIVE["config"] == 2 else (max(cfg["cpu"][0], cores), cfg["cpu"][1])
    n_points = min(n_points, WORKLOAD["n_points"])
    scene = build_scene(n_points, n_frames)
    times = []
    for i in range(args.warmup + args.steps):
        rate, dt = cpu_rate(scene, n_points, cores)
        if i >= args.warmup:
            times.append(dt)
    ms = 1e3 * float(np.mean(times))
    value = n_points * scene.n_particles * n_frames / (ms / 1e3)
    sample = f"{n_points} points x {scene.n_particles} particles x {n_frames} frames of the workload, fork pool over points"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD_NAME, "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------
def run_gpu_arm(args):
    import torch

    import glimpse_b200 as gb
    from glimpse_b200 import _lib, synthetic
    from glimpse_b200.session import Session

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    device = torch.device("cuda", local_rank)
    P, N, T = WORKLOAD["n_points"], WORKLOAD["n_particles"], WORKLOAD["n_frames"]
    if args.small:
        P, T = 64, 12
    if args.points:
        P, args.small = args.points, True
    if args.frames:
        T, args.small = args.frames, True
    scene = build_scene(P * world, T, pinned=True)
    observers, models = synthetic.build(scene, gb)
    tracker = gb.Tracker(observers, seed=20260101)
    datetimes = tracker.datetimes
    matching = tracker.match_datetimes(datetimes)
    image_index = np.array([[-1 if v is None else int(v) for v in row] for row in matching], dtype=np.int32)
    unit = scene.time_unit.total_seconds()
    taus = np.array([dt.total_seconds() / unit for dt in np.diff(datetimes)])
    lo, hi = rank * P, (rank + 1) * P
    mask = np.ones((P, len(observers)), dtype=bool)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------- value: device-resident inputs, CUDA events on the launching stream ----------
    session = Session(tracker, models[lo:hi], image_index, taus, scene.tile_size, mask, point_offset=lo)
    gathered = None
    if dist is not None:
        gathered = [torch.empty((world,) + tuple(session.buf[k].shape), dtype=torch.float64, device=device)
                    for k in ("means", "sig")]

    def one_track(events=None):
        session.buf["status"].zero_()
        if args.per_step_events:
            session.init(0)
            for t in range(1, T):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                session.step(t)
                b.record()
                if events is not None:
                    events.append((a, b))
        else:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            session.run()  # gb_track: every update of every point, asynchronously
            b.record()
            if events is not None:
                events.append((a, b))
        if dist is not None:
            dist.all_gather_into_tensor(gathered[0], session.buf["means"])
            dist.all_gather_into_tensor(gathered[1], session.buf["sig"])

    for _ in range(args.warmup):
        one_track()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    step_events = []
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(args.steps):
        one_track(step_events)
    end.record()
    barrier()
    clocks = sampler.stop()
    dev_ms = max_over_ranks(start.elapsed_time(end)) / args.steps
    kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in step_events]))
    if not args.per_step_events:
        kernel_ms /= (T - 1)  # gb_track = init + templates + (T - 1) updates; the updates are > 99 % of it
    status = session.buf["status"].cpu().numpy()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, session.fetch())  # (rank 0's points; the untimed tracks below reuse the buffers)
    # per-kernel durations of one more (untimed) track: CUDA events around every launch on its own stream
    import ctypes as C
    lib = _lib.load()
    KINDS = ["k_s0p_activity", "k_s2_surface", "k_s3_weights", "k_s4p_resample_propagate", "k_s5p_finalize", "k_init", "k_template", "k_s3b_publish"]

    def kernel_times(sess):
        _lib.check(lib.gb_kernel_timing(1))
        sess.buf["status"].zero_()
        sess.run()
        torch.cuda.synchronize()
        k_ms, k_n = (C.c_double * len(KINDS))(), (C.c_int64 * len(KINDS))()
        _lib.check(lib.gb_kernel_timing_read(k_ms, k_n, len(KINDS)))
        _lib.check(lib.gb_kernel_timing(0))
        return {name: {"ms_per_track": float(k_ms[i]), "launches": int(k_n[i]),
                       "us_per_launch": 1e3 * float(k_ms[i]) / max(1, int(k_n[i]))} for i, name in enumerate(KINDS)}

    kernels, kernels_serial = {}, {}
    session.launches = 0
    if args.mode == "stream" and not args.per_step_events:
        kernels = kernel_times(session)  # production plan: batches overlap on their streams, durations include sharing
    launches_per_track = session.launches
    session.launches = 0
    stats_out = session.fetch()
    if kernels and rank == 0:
        # the same track with all points in one batch on one stream: launches do not overlap, so the per-launch
        # durations are those of each kernel alone (warm caches) — the figures the per-kernel roofline uses
        saved = {k: os.environ.get(k) for k in ("GB_STREAM_SLOTS", "GB_STREAM_BATCH")}
        os.environ["GB_STREAM_SLOTS"], os.environ["GB_STREAM_BATCH"] = "1", str(P)
        try:
            serial = Session(tracker, models[lo:hi], image_index, taus, scene.tile_size, mask, point_offset=lo)
            serial.run()
            torch.cuda.synchronize()
            kernels_serial = kernel_times(serial)
            del serial
        finally:
            for k, v in saved.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
    failed = int((status != 0).sum())
    value = world * P * N * T / (dev_ms / 1e3)
    if launches_per_track:
        launches_per_step = launches_per_track  # counted by gb_track itself
    else:
        nbatch = -(-P // max(1, session.stats["plan"].get("stream_batch", P) or P)) if args.mode == "stream" else 1
        launches_per_step = 2 + (6 * nbatch if args.mode == "stream" else 1) * (T - 1)
    peak, peak_src = hbm_peak()
    achieved = ALGORITHMIC_BYTES_PER_UPDATE * P * N / (kernel_ms / 1e3) / 1e9
    win_w, win_h = session.stats["window_width"], session.stats["window_height"]
    update = {"achieved": achieved, "frac": achieved / peak, "ms": kernel_ms,
              "what": "one update of all points (every kernel and batch), algorithmic bytes / (track time / updates)"}
    dom = kernels_serial.get("k_s4p_resample_propagate")
    if dom and dom["launches"]:
        # dominant kernel: SURVEY.md 8(d)'s 96 B per particle-update x the particles one launch processes
        dom_bytes = ALGORITHMIC_BYTES_PER_UPDATE * P * N
        dom_ach = dom_bytes / (dom["us_per_launch"] * 1e-6) / 1e9
        total_ms = sum(v["ms_per_track"] for v in kernels_serial.values())
        roofline = {"bound": "hbm", "achieved": dom_ach, "peak": peak, "unit": "GB/s", "frac": dom_ach / peak,
                    "traffic": S4P_DRAM_BYTES_PER_PARTICLE * P * N if (not args.small and ACTIVE["config"] == 2) else None,
                    "traffic_source": "constant from the ncu --set full capture of this kernel (profiles/), not measured in this run",
                    "kernel": "k_s4p_resample_propagate", "kernel_ms": dom["us_per_launch"] / 1e3, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": dom_bytes, "share_of_step": dom["ms_per_track"] / total_ms,
                    "measured": "CUDA events around every launch on the launching stream, all points in one batch (no overlap)",
                    "whole_update": update, "kernels_serial": kernels_serial, "kernels": kernels}
    else:
        roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                    "kernel": "one update of all points", "kernel_ms": kernel_ms,
                    "peak_source": peak_src, "algorithmic_bytes_per_launch": ALGORITHMIC_BYTES_PER_UPDATE * P * N}

    # ---------------- e2e: public API, host frames, copies inside the timed region -----------------
    def e2e_once():
        tracker.clear_device_cache()
        return tracker.track(models, tile_size=scene.tile_size)

    e2e_steps = args.steps
    # (the warm-up calls keep ALL their results until the last one is done: a call needs a fresh set of pinned result buffers
    #  whenever every cached set is still referenced, and a first cudaHostAlloc of that set — 2 x 38 MB at 8 GPUs, 8 processes
    #  at once — costs ~50 ms (tools/e2e_steps.py: host_alloc 2 in exactly the slow calls).  Three sets cached here cover the
    #  steady state of a loop that keeps its previous result; `host_alloc_each_rank0` below shows that no timed step allocated.)
    held = [e2e_once() for _ in range(max(3, min(args.warmup, 3)))]
    tracks = held[-1]
    del held
    barrier()

    def host_allocs():
        stats = torch.cuda.host_memory_stats() if hasattr(torch.cuda, "host_memory_stats") else {}
        return int(stats.get("num_host_alloc", 0))

    import gc

    gc.collect()
    gc.disable()  # as timeit does: a cyclic collection over the scene's objects would land in one of the steps
    t0 = time.perf_counter()
    e2e_each, e2e_host, e2e_allocs = [], [], []
    for _ in range(e2e_steps):
        t1, a1 = time.perf_counter(), host_allocs()
        tracks = e2e_once()
        e2e_each.append(1e3 * (time.perf_counter() - t1))  # track() returns host arrays: the device is idle again
        e2e_allocs.append(host_allocs() - a1)
        e2e_host.append({k: round(v, 2) for k, v in tracker.last_run.get("host_ms", {}).items()})
    torch.cuda.synchronize()
    # the mean of the steps is the value (what a user sees); every step time is in ms_each, the median beside it
    e2e_mean_s = max_over_ranks((time.perf_counter() - t0) / e2e_steps)
    e2e_median_s = max_over_ranks(float(np.median(e2e_each)) / 1e3)
    gc.enable()
    e2e_value = world * P * N * T / e2e_mean_s
    e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(tracker.last_run["h2d_bytes"]),
           "d2h_bytes_per_step": int(tracker.last_run["d2h_bytes"]), "ms_per_step": 1e3 * e2e_mean_s, "steps": e2e_steps,
           "ms_each": e2e_each, "median_ms_per_step": 1e3 * e2e_median_s, "aggregate": "mean of steps (max over ranks)",
           "host_ms_last_step": {k: round(v, 2) for k, v in tracker.last_run.get("host_ms", {}).items()},
           "host_ms_each_rank0": e2e_host, "host_alloc_each_rank0": e2e_allocs}
    v_err = float(np.nanmedian(np.abs(tracks.vxyz[:, -1, 0] - scene.truth_velocity[0])))

    # ---------------- CPU baseline (rank 0, N = 1): bounded sample of the same workload ------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        sub_points, sub_frames = CONFIGS[ACTIVE["config"]]["cpu"]  # 10-30 s on one core
        sub_points = min(sub_points, P)
        sub = build_scene(sub_points, sub_frames)
        os.environ.setdefault("OMP_NUM_THREADS", "1")
        rate, dt = cpu_rate(sub, sub_points, 1)
        cpu = {"value": rate, "unit": UNIT, "cores": 1, "kind": "port", "seconds": dt,
               "sample": f"{sub_points} points x {N} particles x {sub_frames} frames of the workload (oracle/tracker_oracle.py)"}

    # ---------------- sharding check, strong scaling, the other named shapes -------------------------
    extra = {}
    if not args.small and ACTIVE["config"] == 2 and not args.no_side:
        extra = side_records(gb, synthetic, scene, world, rank, device, max_over_ranks, barrier, hbm_peak()[0], args)
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {
                "workload": WORKLOAD_NAME if not args.small else f"SMALL smoke variant: {P} points x {N} particles x {T} frames",
                "points_per_gpu": P, "particles": N, "frames": T, "rng": "philox (device)", "mode": args.mode,
                "cache": "inputs larger than L2 (particle state 2 x %.0f MB per GPU, no flush needed)" % (P * N * 48 / 1e6),
                "plan": session.stats["plan"],
                "search_window_px": {"median_w": float(np.median(win_w)) if len(win_w) else None,
                                     "median_h": float(np.median(win_h)) if len(win_h) else None,
                                     "p90_w": float(np.percentile(win_w, 90)) if len(win_w) else None,
                                     "p99_w": float(np.percentile(win_w, 99)) if len(win_w) else None,
                                     "max_w": int(win_w.max()) if len(win_w) else None,
                                     "max_h": int(win_h.max()) if len(win_h) else None},
                "failed_points": failed, "median_abs_velocity_error_m_per_day": v_err,
            },
            "roofline": roofline,
            "cpu_baseline": cpu,
            "e2e": e2e,
            "gpu_launches": launches_per_step * args.steps,
            "clocks": clocks,
        }
        line.update(extra)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def side_records(gb, synthetic, main_scene, world, rank, device, max_over_ranks, barrier, peak, args):
    """Three records beside the headline (config 2) line:
    result_crc  CRC-32 of the means and sigmas of a fixed 64-point problem tracked through the public API, sharded over the
                ranks of this run: the same number at every N (the device draws are keyed by the global point index), and
                the same as result_crc_one_gpu, the problem tracked on one GPU in the same run.
    strong      strong scaling: a fixed 8 000 points of the workload split over the ranks, end to end (frames uploaded once
                per box and shared over NVLink, one gather of the results).
    configs     one end-to-end track() each of BASELINE.json's other single-GPU shapes (rank 0's GPU only), with the frames
                already on the device (the second call), as particle-updates/s and as fraction of the HBM roofline."""
    import zlib

    import torch

    out = {}
    small = synthetic.nadir_scene(seed=77, n_points=64, n_particles=2000, n_frames=8, imgsz=(600, 400))
    observers, models = synthetic.build(small, gb)
    def crc_of(tracks):
        crc = zlib.crc32(np.ascontiguousarray(tracks.means).tobytes())
        return "%08x" % zlib.crc32(np.ascontiguousarray(tracks.sigmas).tobytes(), crc)

    out["result_crc"] = crc_of(gb.Tracker(observers, seed=777).track(models, tile_size=small.tile_size))
    # the same problem on this rank's GPU alone, and a checksum of its (host-generated) frames: the three numbers of runs on
    # different boxes can only be compared if the frames agree (SciPy's filter may round differently on another CPU)
    out["result_crc_one_gpu"] = crc_of(gb.Tracker(observers, seed=777, distributed=False).track(models, tile_size=small.tile_size))
    out["result_crc_frames"] = "%08x" % zlib.crc32(b"".join(np.ascontiguousarray(f).tobytes() for f in small.observers[0].frames))
    # ---- strong scaling
    total = 8000
    kw = dict(WORKLOAD)
    kw.update(n_points=total, n_frames=2)
    strong = synthetic.nadir_scene(**dict(kw, n_frames=len(main_scene.observers[0].frames)))
    strong.observers[0].frames = main_scene.observers[0].frames  # the same (pinned) frames: they do not depend on the points
    observers, models = synthetic.build(strong, gb)
    tracker = gb.Tracker(observers, seed=20260102)
    times = []
    for i in range(3):
        tracker.clear_device_cache()
        barrier()
        t0 = time.perf_counter()
        tracks = tracker.track(models, tile_size=strong.tile_size)
        torch.cuda.synchronize()
        if i:
            times.append(time.perf_counter() - t0)
    sec = max_over_ranks(float(np.mean(times)))
    T = len(strong.datetimes)
    out["strong"] = {"points_total": total, "particles": strong.n_particles, "frames": T, "n_gpus": world, "ms_per_track": 1e3 * sec,
                     "value": total * strong.n_particles * T / sec, "unit": UNIT, "failed_points": int(sum(e is not None for e in tracks.errors)),
                     "what": "end-to-end Tracker.track of a FIXED 8000 points sharded over the ranks (host frames, mean of 2)"}
    del tracker, tracks, observers, models, strong
    # ---- the other named shapes, one GPU each run (rank 0 reports)
    configs = {}
    if rank == 0 or world == 1:
        saved = ACTIVE["config"]
        for number in (1, 3, 4):
            select_config(number)
            try:
                cfg = CONFIGS[number]
                scene = build_scene(cfg["scene"]["n_points"], cfg["scene"]["n_frames"])
                observers, models = synthetic.build(scene, gb)
                tracker = gb.Tracker(observers, seed=20260100 + number, distributed=False)
                best = None
                for rep in range(3):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    tracks = tracker.track(models, tile_size=scene.tile_size)
                    torch.cuda.synchronize()
                    dt = time.perf_counter() - t0
                    if rep:
                        best = dt if best is None else min(best, dt)
                P, N, T = len(models), scene.n_particles, len(scene.datetimes)
                rate = P * N * T / best
                win = tracker.last_run["window_width"]
                configs[f"config{number}"] = {
                    "workload": cfg["name"], "value": rate, "unit": UNIT, "ms_per_track": 1e3 * best,
                    "algorithmic_bytes_per_update": cfg["bytes"],
                    "roofline": {"bound": "hbm", "achieved": rate * cfg["bytes"] / 1e9, "peak": peak, "unit": "GB/s",
                                 "frac": rate * cfg["bytes"] / 1e9 / peak, "what": "whole track() call, frames resident"},
                    "failed_points": int(sum(e is not None for e in tracks.errors)),
                    "median_abs_velocity_error_m_per_day": float(np.nanmedian(np.abs(tracks.vxyz[:, -1, 0] - scene.truth_velocity[0]))),
                    "search_window_px": {"median_w": float(np.median(win)) if len(win) else None, "max_w": int(win.max()) if len(win) else None},
                    "kernel_launches": int(tracker.last_run["kernel_launches"]),
                }
                del tracker, tracks, observers, models, scene
                torch.cuda.empty_cache()
            except Exception as exc:  # a side record must not take the headline down
                configs[f"config{number}"] = {"error": repr(exc)[:300]}
        select_config(saved)
    barrier()
    out["configs"] = configs
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="glimpse_b200", choices=["glimpse_b200", "reference"])
    ap.add_argument("--mode", default="stream", choices=["stream"])
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 3, 4],
                    help="BASELINE.json config (1-based; the default 2 is the one the metric is quoted on)")
    ap.add_argument("--no-side", action="store_true", help="skip the sharding check / strong scaling / other shapes records")
    ap.add_argument("--small", action="store_true", help="tiny variant for smoke-testing the script (not a bench value)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--per-step-events", action="store_true", help="drive the updates one gb_track_step at a time with CUDA events around each")
    ap.add_argument("--points", type=int, default=0, help="override points per GPU (profiling only; not a bench value)")
    ap.add_argument("--frames", type=int, default=0, help="override frame count (profiling only; not a bench value)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the results of the GPU arm")
    select_config(args.config)
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
