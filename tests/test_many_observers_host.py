"""CPU-side checks of calls with more than eight observers: the count of observers with a frame at the same time, the
refusal of more than eight of them, the session's memory estimate and the C ABI's argument checks."""
import ctypes as C

import numpy as np
import pytest

from glimpse_b200 import synthetic


def test_observer_slots_count_the_observers_with_a_frame_at_one_time():
    from glimpse_b200.session import observer_slots, plan_slots

    assert observer_slots(np.array([[0, -1, 3], [-1, -1, -1], [1, 2, -1]])) == 2
    assert observer_slots(np.full((4, 20), -1)) == 0
    grid = np.full((5, 12), -1)
    grid[1, [2, 7, 10]] = 0
    grid[3, [0, 11]] = 4
    assert observer_slots(grid) == 3
    grid[2, :9] = 1
    assert observer_slots(grid) == 9
    # one slot per observer up to eight observers, whatever their frames; beyond, the count above (at least one)
    assert plan_slots(np.full((3, 5), -1)) == 5
    assert plan_slots(np.zeros((3, 8))) == 8
    assert plan_slots(np.full((3, 9), -1)) == 1
    grid[2, :9] = -1
    assert plan_slots(grid) == 3


def test_nine_observers_at_one_time_are_refused_before_device_work(monkeypatch):
    """Fourteen observers; at time index 4 nine of them have a frame.  The refusal names that time and comes before any
    device work (here there is no device: reaching it would fail differently)."""
    import glimpse_b200 as gb
    from glimpse_b200 import _lib

    def no_device():
        raise AssertionError("device work started")

    monkeypatch.setattr(_lib, "require_cuda", no_device)
    scene = synthetic.nadir_scene(seed=3, n_points=2, n_particles=64, n_frames=7, imgsz=(160, 120), margin_px=40)
    base = scene.observers[0]
    schedule = [{0, 1, 3, 4}, {1, 2}, {2, 3, 4}, {0, 5}, set(range(5, 14)), {6, 7, 8, 13}, {9, 10, 11, 12}]
    scene.observers = [synthetic.ObserverScene([base.frames[t] for t in range(7) if o in schedule[t]],
                                               np.array([base.cams[t] for t in range(7) if o in schedule[t]]),
                                               [base.datetimes[t] for t in range(7) if o in schedule[t]]) for o in range(14)]
    observers, models = synthetic.build(scene, gb)
    with pytest.raises(NotImplementedError, match=r"9 observers have an image at time index 4.*at most 8"):
        gb.Tracker(observers, rng="numpy").track(models, tile_size=scene.tile_size)
    # eight at that time: the check passes and the call goes on to the device
    scene.observers[13] = synthetic.ObserverScene(base.frames[5:7], np.array(base.cams[5:7]), base.datetimes[5:7])
    observers, models = synthetic.build(scene, gb)
    with pytest.raises(AssertionError, match="device work started"):
        gb.Tracker(observers, rng="numpy").track(models, tile_size=scene.tile_size)


def test_session_bytes_size_the_scratch_by_slots_and_the_templates_by_observers():
    from glimpse_b200 import _lib
    from glimpse_b200.session import session_bytes

    lib = _lib.load()
    S = _lib.GB_MODE_STREAM
    shape = dict(N=1000, T=40, tw=15, th=15, return_covariances=False, return_particles=False)
    twelve = session_bytes(lib, S, 0, 50, O=12, slots=3, **shape)
    three = session_bytes(lib, S, 0, 50, O=3, **shape)
    # per point and observer: three template arrays of w x h doubles and 40 B of template scalars; T flag bytes and window sizes
    per_observer = 3 * 15 * 15 * 8 + 40 + 40 * 9
    assert twelve - three == 50 * 9 * per_observer
    assert three - 50 * 3 * per_observer == session_bytes(lib, S, 0, 50, O=1, slots=3, **shape) - 50 * per_observer
    assert session_bytes(lib, S, 0, 50, O=3, slots=3, **shape) == three
    with pytest.raises(RuntimeError):  # twelve observers cannot have a slot each
        session_bytes(lib, S, 0, 50, O=12, **shape)


def desc_with(O, T, index, plan_slots, N=4):
    """A descriptor whose argument checks pass up to the observer slots (device pointers are never dereferenced by them).
    N = 8 particles against a plan for 4: a descriptor that passes the slot checks fails the next one, 'plan does not cover
    N particles', before any device work."""
    from glimpse_b200 import _lib

    lib = _lib.load()
    d = _lib.gb_track_desc()
    d.P, d.N, d.T, d.O, d.tile_w, d.tile_h = 1, N, T, O, 15, 15
    assert lib.gb_step_plan(4, 15, 15, 1, plan_slots, 0, _lib.GB_MODE_STREAM, C.byref(d.plan)) == 0
    fake = 1 << 20
    for name in ("images", "mask", "first", "last", "motion", "surfaces", "state_a", "state_b", "means", "sigmas", "status",
                 "status_time", "obs_flags", "tmpl_tile", "tmpl_values", "tmpl_quantiles", "tmpl_nvalues", "tmpl_box", "tmpl_duv",
                 "scratch", "init_normals", "step_normals", "uniforms"):
        setattr(d, name, fake)
    images = (_lib.gb_image * (O * T))()
    for im in images:
        im.nchan = 1
    offsets = np.arange(O, dtype=np.int32) * T
    index = np.ascontiguousarray(index, dtype=np.int32)
    d.images_host, d.image_offset_host, d.image_index_host = C.addressof(images), offsets.ctypes.data, index.ctypes.data
    return lib, d, (images, offsets, index)


def entry_points(lib, d):
    return {"gb_track": lambda: lib.gb_track(C.byref(d), None, None),
            "gb_track_step": lambda: lib.gb_track_step(C.byref(d), 1, None, None),
            "gb_track_init": lambda: lib.gb_track_init(C.byref(d), 0, None)}


def test_track_entry_points_check_the_observer_slots():
    T, O = 4, 12
    index = np.full((T, O), -1)
    index[0, [0, 1, 4]] = 0
    index[1, [2, 7, 10]] = 1
    index[2, [3, 5]] = 2
    index[3, 11] = 3
    # a plan with fewer slots than the three observers of time 1: invalid
    lib, d, keep = desc_with(O, T, index, plan_slots=2)
    for name, call in entry_points(lib, d).items():
        assert call() == -1, name
        assert b"observers with a frame at the same time" in lib.gb_last_error(), name
    # three slots, or more: the slot checks pass
    for slots in (3, 8):
        lib, d, keep = desc_with(O, T, index, plan_slots=slots, N=8)
        for name, call in entry_points(lib, d).items():
            assert call() == -1, (name, slots)
            assert b"plan does not cover N particles" in lib.gb_last_error(), (name, slots)
    # nine observers with a frame at time 2: no plan has room for them
    index[2, :9] = 2
    lib, d, keep = desc_with(O, T, index, plan_slots=8)
    for name, call in entry_points(lib, d).items():
        assert call() == -3, name
        assert b"more than 8 observers" in lib.gb_last_error(), name


def test_up_to_eight_observers_keep_one_slot_each():
    T = 3
    for O in (1, 3, 8):
        index = np.full((T, O), -1)
        index[:, 0] = 0  # one observer with frames: a call of up to eight observers still plans one slot per observer
        for slots in range(1, 9):
            lib, d, keep = desc_with(O, T, index, plan_slots=slots, N=8)
            for name, call in entry_points(lib, d).items():
                assert call() == -1, (O, slots, name)
                expect = b"plan does not cover N particles" if slots == O else b"streaming plan does not match the descriptor"
                assert expect in lib.gb_last_error(), (O, slots, name, lib.gb_last_error())
    # the plan itself still takes 1 to 8 slots
    from glimpse_b200 import _lib

    plan = _lib.gb_plan()
    assert lib.gb_step_plan(4, 15, 15, 1, 9, 0, _lib.GB_MODE_STREAM, C.byref(plan)) == -1
    assert lib.gb_step_plan(4, 15, 15, 1, 0, 0, _lib.GB_MODE_STREAM, C.byref(plan)) == -1


def test_observer_flag_values_match_the_header():
    """obs_flags values the Python layer compares with (GB_OBS_*) are those of include/glimpse_b200.h."""
    import os
    import re

    from glimpse_b200 import _lib

    header = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "glimpse_b200.h")).read()
    values = {name: int(v) for name, v in re.findall(r"#define (GB_OBS_\w+) (\d+)", header)}
    assert values["GB_OBS_NO_IMAGE"] == _lib.GB_OBS_NO_IMAGE
    assert values["GB_OBS_OUT_OF_FRAME"] == _lib.GB_OBS_OUT_OF_FRAME
