"""Twelve observers with three of them active at every time, against the same three stations as three observers, on the
config-2 frames (4288 x 2848 uint8, full distortion): 1 000 points x 10 000 particles x 50 frames, one GPU.

    python tools/many_observers_bench.py [--reps 5] [--out DIR]

Three stations see every frame.  The twelve-observer call cuts each station's frames into four runs of consecutive times,
one observer per run (a station that was moved or re-calibrated becomes a new observer): three observers have a frame at
every time, so the plan has three slots.  Per time step both calls do the same window work; the twelve-observer call also
cuts a template whenever a new observer starts.  One JSON line per call: ms per track (median of --reps timed gb_track calls
after one warm-up, CUDA events on the launching stream) and G particle-updates/s.  The first line names the card and its
power limit.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def stations(base, runs):
    """Three stations over the base frames, each cut into ``runs`` observers of consecutive times."""
    from glimpse_b200 import synthetic

    T = len(base.frames)
    cuts = np.linspace(0, T, runs + 1).astype(int)
    out = []
    for k in range(3):
        for a, b in zip(cuts[:-1], cuts[1:]):
            out.append(synthetic.ObserverScene(base.frames[a:b], base.cams[a:b].copy(), list(base.datetimes[a:b]), sigma=0.3 + 0.05 * k))
    return out


def one_call(name, scene, runs, args, gb, torch):
    from glimpse_b200 import synthetic
    from glimpse_b200.session import Session, plan_slots

    base = scene.observers[0]
    call = synthetic.Scene(stations(base, runs), scene.points, scene.motion, scene.n_particles, scene.tile_size, scene.time_unit)
    observers, models = synthetic.build(call, gb)
    tracker = gb.Tracker(observers, seed=20260101)
    datetimes = tracker.datetimes
    index = np.array([[-1 if v is None else int(v) for v in row] for row in tracker.match_datetimes(datetimes)], dtype=np.int32)
    unit = scene.time_unit.total_seconds()
    taus = np.array([dt.total_seconds() / unit for dt in np.diff(datetimes)])
    P, N, T, O = args.points, args.particles, len(datetimes), len(observers)
    session = Session(tracker, models, index, taus, scene.tile_size, np.ones((P, O), dtype=bool))
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
    out = {"call": name, "observers": O, "slots": int(plan_slots(index)), "points": P, "particles": N, "frames": T,
           "failed_points": int((res["status"] != 0).sum()), "ms_per_track": round(ms, 2), "ms_all": [round(t, 2) for t in times],
           "G_particle_updates_per_s": round(P * N * T / (ms / 1e3) / 1e9, 3)}
    del session
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--points", type=int, default=1000)
    ap.add_argument("--particles", type=int, default=10000)
    ap.add_argument("--frames", type=int, default=50)
    ap.add_argument("--out", default=None, help="also write the lines to DIR/many_observers_bench.jsonl")
    args = ap.parse_args()
    import torch

    import glimpse_b200 as gb
    from glimpse_b200 import synthetic

    if not torch.cuda.is_available():
        raise SystemExit("this benchmark needs a CUDA device")
    lines = [{"card": card(), "query": "name, power.limit, clocks.max.sm"}]
    print(json.dumps(lines[0]), flush=True)
    scene = synthetic.nadir_scene(seed=2, n_points=args.points, n_particles=args.particles, n_frames=args.frames, imgsz=(4288, 2848),
                                  velocity_sigma=0.2, margin_px=200)
    # alternating, twice each: the spread between repeats of one call bounds what the difference between the calls can say
    for name, runs in (("12 observers, 3 active", 4), ("3 observers", 1)) * 2:
        lines.append(one_call(name, scene, runs, args, gb, torch))
        print(json.dumps(lines[-1]), flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "many_observers_bench.jsonl"), "w") as f:
            f.writelines(json.dumps(x) + "\n" for x in lines)


if __name__ == "__main__":
    main()
