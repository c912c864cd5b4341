"""Raster.viewshed on the device (gb_viewshed): seeded square DEMs (scenes.viewshed_large_case) seen from a point near their
middle, curvature and refraction corrected.  For every side: end-to-end time of Raster.viewshed (host array in, boolean array out),
device time of the kernels alone (CUDA events, DEM resident, median of 5), the work-buffer bytes and the largest ring.  The first
line names the card and its power limit.

    python tools/viewshed_bench.py [side ...] [--eye-above M] [--ab LIB]

--eye-above: the eye M metres above the terrain under it (default 30, the full-size golden's).  --ab LIB: also time another
build of the library (same C ABI, e.g. the parent commit's) on the same resident inputs, alternating with this one, and check
that both give the same cells."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import glimpse_b200 as gb  # noqa: E402
from glimpse_b200 import _lib  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "tests"))
import scenes  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("sides", nargs="*", type=int, default=[2000])
ap.add_argument("--eye-above", type=float, default=30.0)
ap.add_argument("--ab", default=None)
ap.add_argument("--rounds", type=int, default=6)
args = ap.parse_args()

torch = _lib.require_cuda()
lib = _lib.load()
dev = torch.device("cuda", 0)
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
print(json.dumps({"card": torch.cuda.get_device_name(0), "nvidia_smi": smi.stdout.strip()}), flush=True)

other = None
if args.ab:
    other = C.CDLL(args.ab)
    for name in ("gb_viewshed_work_bytes", "gb_viewshed"):
        getattr(other, name).restype, getattr(other, name).argtypes = _lib.SIGNATURES[name]


def device_ms(L, side, z_d, x_d, y_d, origin, max_rings, reps=5):
    nbytes = int(L.gb_viewshed_work_bytes(side, side, max_rings))
    work = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    out = torch.empty(side * side, dtype=torch.uint8, device=dev)
    corr = (C.c_double * 2)(6.3781e6, 0.13)
    ms = []
    for _ in range(reps + 1):  # (the first is a warm-up)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        _lib.check(L.gb_viewshed(z_d.data_ptr(), side, side, x_d.data_ptr(), y_d.data_ptr(), 10.0, (C.c_double * 3)(*origin), corr,
                                 max_rings, work.data_ptr(), nbytes, out.data_ptr(), torch.cuda.current_stream().cuda_stream))
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    assert int(work[:4].cpu().numpy().view(np.int32)[0]) == 0
    return float(np.median(ms[1:])), nbytes, out.cpu().numpy().reshape(side, side).astype(bool)


for side in args.sides:
    case = scenes.viewshed_large_case(side)
    z = case["z"]
    origin = case["origin"][:2] + (case["origin"][2] - 30.0 + args.eye_above,)
    raster = gb.Raster(z, x=case["xlim"], y=case["ylim"])
    vis = raster.viewshed(origin, correction=True)  # warm-up (module load, allocator)
    t0 = time.perf_counter()
    vis = raster.viewshed(origin, correction=True)
    e2e_ms = 1e3 * (time.perf_counter() - t0)
    x, y = raster.x, raster.y
    max_rings = int(np.hypot(side, side)) + 8
    z_d, x_d, y_d = (torch.from_numpy(np.array(v, dtype=float, order="C", copy=True)).to(dev) for v in (z, x, y))
    sizes = np.zeros(int(np.hypot(side, side)) + 8, dtype=np.int64)
    for r0 in range(0, side, 500):  # (ring sizes, a block of rows at a time)
        rings = (np.hypot(*np.meshgrid(x - origin[0], y[r0:r0 + 500] - origin[1])) * (1 / 10.0) + 0.5).astype(int)
        sizes += np.bincount(rings.ravel(), minlength=sizes.size)
    res = {"what": f"Raster.viewshed of a {side} x {side} DEM (curvature / refraction corrected), eye {args.eye_above:g} m above "
                   "a point near the middle", "cells": side * side, "largest_ring": int(sizes.max()),
           "e2e_ms": e2e_ms, "visible_fraction": float(vis.mean())}
    if other is None:
        ms, nbytes, got = device_ms(lib, side, z_d, x_d, y_d, origin, max_rings)
        assert np.array_equal(got, vis)
        res.update(device_ms=ms, work_bytes=nbytes, Mcells_per_s_device=side * side / ms / 1e3)
    else:  # alternate the two builds, each round the median of 5
        mine, theirs = [], []
        for _ in range(args.rounds):
            ms, nbytes, got = device_ms(lib, side, z_d, x_d, y_d, origin, max_rings)
            mine.append(ms)
            assert np.array_equal(got, vis)
            ms, nb_other, got = device_ms(other, side, z_d, x_d, y_d, origin, max_rings)
            theirs.append(ms)
            assert np.array_equal(got, vis), "the two builds differ"
        res.update(device_ms_rounds=mine, other_device_ms_rounds=theirs, device_ms=float(np.median(mine)),
                   other_device_ms=float(np.median(theirs)), work_bytes=nbytes, other_work_bytes=nb_other)
    print(json.dumps(res), flush=True)
    del z_d, x_d, y_d
    torch.cuda.empty_cache()
