"""CPU-side checks of templates above 1024 pixels: the GB_PLAN_LARGE_TEMPLATES plan flag, the Python layer's use of it and
its refusal beyond 128 pixels a side, and the tolerance the GPU tests of these sizes rely on."""
import ctypes as C
import warnings

import numpy as np
import pytest

import helpers
from glimpse_b200 import synthetic
from oracle import tracker_oracle as orc


def plan(tw, th, flags, margin=191):
    from glimpse_b200 import _lib

    lib = _lib.load()
    out = _lib.gb_plan()
    rc = lib.gb_step_plan_ex(1000, tw, th, 10, 1, flags, _lib.GB_MODE_STREAM, margin, C.byref(out))
    return rc, out, lib


def test_plan_flag_semantics():
    from glimpse_b200 import _lib

    large = _lib.GB_PLAN_LARGE_TEMPLATES
    assert large == 2
    rc, _, lib = plan(40, 40, 0)
    assert rc == -3 and b"1024" in lib.gb_last_error()
    sizes = []
    for tw, th in ((40, 40), (64, 48), (128, 128)):
        rc, p, _ = plan(tw, th, large)
        assert rc == 0, (tw, th)
        assert p.max_template == tw * th
        sizes.append(p.surf_bytes)
    assert sizes[0] < sizes[1] < sizes[2]
    # both flags together (ranked frames) and odd sizes
    assert plan(127, 33, large | _lib.GB_PLAN_RANKED_FRAMES)[0] == 0
    for tw, th in ((129, 8), (8, 129), (129, 129)):
        rc, _, lib = plan(tw, th, large)
        assert rc == -3, (tw, th)
        assert b"128" in lib.gb_last_error()
    assert plan(15, 15, 4)[0] == -1
    assert plan(40, 40, large | 4)[0] == -1
    # up to 1024 pixels the flag changes nothing in the plan
    for tw, th in ((15, 15), (32, 32), (200, 5)):
        a, b = plan(tw, th, 0)[1], plan(tw, th, large)[1]
        assert bytes(a) == bytes(b), (tw, th)


def test_session_bytes_large_template():
    from glimpse_b200 import _lib
    from glimpse_b200.session import session_bytes

    lib = _lib.load()
    shape = dict(N=1000, T=5, O=1, return_covariances=False, return_particles=False)
    small = session_bytes(lib, [], None, 10, tw=32, th=32, **shape)
    large = session_bytes(lib, [], None, 10, tw=64, th=64, **shape)
    assert large > small > 0


def test_track_refuses_sides_above_128_before_device_work(monkeypatch):
    import glimpse_b200 as gb
    from glimpse_b200 import _lib

    def no_cuda(*args, **kwargs):
        raise AssertionError("the device was touched")

    monkeypatch.setattr(_lib, "require_cuda", no_cuda)
    scene = synthetic.nadir_scene(seed=1, n_points=2, n_particles=50, n_frames=3, imgsz=(320, 240))
    observers, models = synthetic.build(scene, gb)
    tracker = gb.Tracker(observers, rng="numpy")
    for size in ((129, 129), (129, 9), (9, 129)):
        with pytest.raises(NotImplementedError, match="128"):
            tracker.track(models, tile_size=size)


def test_oracle_sse_at_128_is_within_tolerance_of_exact_ssd():
    """OpenCV's float32 matchTemplate (what the reference computes) against an exact float64 SSD of the same tiles for a
    128 x 128 template: within the 5e-5 the GPU tests allow between the device and OpenCV."""
    scene = synthetic.nadir_scene(seed=61, n_points=2, n_particles=200, n_frames=5, imgsz=(600, 400), tile_size=(128, 128),
                                  margin_px=150)
    obs, models, taus, idx = helpers.oracle_inputs(scene)
    np.random.seed(6161)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        res = orc.track(obs, models, taus, idx, tile_size=scene.tile_size, trace=True)
    tiles = {(k // len(obs), int(t["obs"])): t["tile"] for k, t in enumerate(res.templates)}
    steps = [s for s in res.trace if "obs" in s]
    per = len(steps) // len(models)
    worst, n = 0.0, 0
    for i, s in enumerate(steps):
        for o, rec in s["obs"].items():
            exact = orc.ssd_surface(rec["search"], tiles[(i // per, int(o))], exact=True)
            worst = max(worst, float(np.max(np.abs(rec["sse"] - exact) / np.maximum(exact, 1e-3))))
            n += 1
    assert n >= 4
    assert worst <= 5e-5, worst
