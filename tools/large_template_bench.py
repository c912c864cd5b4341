"""Templates of 15 to 128 px on the config-2 frames (4288 x 2848 uint8, full distortion): 1 000 points x 10 000 particles x
50 frames per tile size, device-resident inputs (one GPU).

    python tools/large_template_bench.py [--sizes 15,31,33,47,63,95,128] [--reps 3] [--dtype uint8|uint16] [--out DIR]

For every size, one JSON line: ms per track (median of --reps timed gb_track calls after one warm-up, CUDA events on the
launching stream), G particle-updates/s, us per launch of every kernel (gb_kernel_timing, production plan: batches overlap on
their streams), the search-window sizes over the track, the share of windows per k_s2_surface organisation (dump_clocks of
the last update re-run through gb_track_step), and the SSD rate: sum of M_u M_v w h pixel pairs over the track's
k_s2_surface time.  The first line names the card and its power limit.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

KINDS = ["k_s0p_activity", "k_s2_surface", "k_s3_weights", "k_s4p_resample_propagate", "k_s5p_finalize", "k_init", "k_template",
         "k_s3b_publish"]
ORGS = {1: "interleaved", 2: "planar", 3: "staged", 0: "global"}


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def one_size(size, args, gb, torch):
    from glimpse_b200 import _lib, synthetic
    from glimpse_b200.session import Session

    scene = synthetic.nadir_scene(seed=2, n_points=args.points, n_particles=args.particles, n_frames=args.frames, imgsz=(4288, 2848),
                                  velocity_sigma=0.2, margin_px=200, tile_size=(size, size))
    if args.dtype == "uint16":  # ranked frames: 200 sub-levels per grey level (k_template ranks the template's grey values)
        rng = np.random.RandomState(17)
        for obs in scene.observers:
            obs.frames = [f.astype(np.uint16) * 200 + rng.randint(0, 200, f.shape).astype(np.uint16) for f in obs.frames]
    observers, models = synthetic.build(scene, gb)
    tracker = gb.Tracker(observers, seed=20260101)
    datetimes = tracker.datetimes
    image_index = np.array([[-1 if v is None else int(v) for v in row] for row in tracker.match_datetimes(datetimes)], dtype=np.int32)
    unit = scene.time_unit.total_seconds()
    taus = np.array([dt.total_seconds() / unit for dt in np.diff(datetimes)])
    P, N, T = args.points, args.particles, args.frames
    session = Session(tracker, models, image_index, taus, scene.tile_size, np.ones((P, 1), dtype=bool))
    session.buf["status"].zero_()
    session.run()  # warm-up
    torch.cuda.synchronize()
    times = []
    for _ in range(args.reps):
        session.buf["status"].zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        session.run()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    ms = float(np.median(times))
    res = session.fetch()
    failed = int((res["status"] != 0).sum())
    lib = _lib.load()
    _lib.check(lib.gb_kernel_timing(1))
    session.buf["status"].zero_()
    session.run()
    torch.cuda.synchronize()
    k_ms, k_n = (C.c_double * len(KINDS))(), (C.c_int64 * len(KINDS))()
    _lib.check(lib.gb_kernel_timing_read(k_ms, k_n, len(KINDS)))
    _lib.check(lib.gb_kernel_timing(0))
    kernels = {name: {"ms_per_track": round(float(k_ms[i]), 3), "launches": int(k_n[i]),
                      "us_per_launch": round(1e3 * float(k_ms[i]) / max(1, int(k_n[i])), 2)} for i, name in enumerate(KINDS)}
    res = session.fetch()
    w, h = session.stats["window_width"].astype(np.int64), session.stats["window_height"].astype(np.int64)
    pairs = float(np.sum((w - size + 1) * (h - size + 1)) * size * size)
    s2_ms = float(k_ms[KINDS.index("k_s2_surface")])
    # organisations of the last update's windows
    clocks = torch.full((P, 1, 16), -1, dtype=torch.int64, device=session.device)
    io = _lib.gb_stage_io()
    io.dump_clocks = clocks.data_ptr()
    session.step(T - 1, io)
    torch.cuda.synchronize()
    c = clocks.cpu().numpy()[:, 0]
    ran = c[:, 7] > 0
    orgs = {ORGS[k]: round(float(np.mean(c[ran, 10] == k)), 4) for k in ORGS} if ran.any() else {}
    out = {
        "tile": size, "dtype": args.dtype, "points": P, "particles": N, "frames": T, "failed_points": failed,
        "ms_per_track": round(ms, 2), "ms_all": [round(t, 2) for t in times],
        "G_particle_updates_per_s": round(P * N * T / (ms / 1e3) / 1e9, 3),
        "plan": {"tile_bytes": int(session.plan.tile_bytes), "surf_bytes": int(session.plan.surf_bytes)},
        "kernels": kernels,
        "windows": {"n": int(len(w)), "width_p5_p50_p95_max": [int(np.percentile(w, q)) for q in (5, 50, 95, 100)] if len(w) else [],
                    "height_p5_p50_p95_max": [int(np.percentile(h, q)) for q in (5, 50, 95, 100)] if len(h) else []},
        "organisation_share_last_update": orgs,
        "ssd_pairs": pairs, "ssd_G_pairs_per_s": round(pairs / (s2_ms / 1e3) / 1e9, 1) if s2_ms > 0 else None,
    }
    del session
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="15,31,33,47,63,95,128")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--points", type=int, default=1000)
    ap.add_argument("--particles", type=int, default=10000)
    ap.add_argument("--frames", type=int, default=50)
    ap.add_argument("--dtype", default="uint8", choices=["uint8", "uint16"], help="pixel type of the frames")
    ap.add_argument("--out", default=None, help="also write the lines to DIR/large_template_bench_<dtype>.jsonl")
    args = ap.parse_args()
    import torch

    import glimpse_b200 as gb

    if not torch.cuda.is_available():
        raise SystemExit("this benchmark needs a CUDA device")
    lines = [{"card": card(), "query": "name, power.limit, clocks.max.sm"}]
    print(json.dumps(lines[0]), flush=True)
    for size in (int(s) for s in args.sizes.split(",")):
        lines.append(one_size(size, args, gb, torch))
        print(json.dumps(lines[-1]), flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, f"large_template_bench_{args.dtype}.jsonl"), "w") as f:
            f.writelines(json.dumps(x) + "\n" for x in lines)


if __name__ == "__main__":
    main()
