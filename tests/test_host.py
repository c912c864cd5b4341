"""CPU-side checks: the C-ABI library loads and exports every declared symbol, the ctypes mirrors
match the header's layout, and the host logic of the Tracker (time matching, spans, sharding,
final gather over gloo) behaves like the reference."""
import ctypes as C
import datetime
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "glimpse_b200.h")


def test_library_exports_every_declared_symbol():
    from glimpse_b200 import _lib, build

    build.build()
    lib = _lib.load()
    text = open(HEADER).read()
    declared = set(re.findall(r"^\s*(?:int|int64_t|const char\*)\s+(gb_\w+)\s*\(", text, flags=re.M))
    assert declared, "no declarations parsed"
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.gb_version() == 1
    # the library was compiled with the layouts the ctypes mirror declares
    for which, struct in enumerate(_lib.STRUCTS):
        assert lib.gb_struct_size(which) == C.sizeof(struct), struct.__name__
    assert lib.gb_struct_size(len(_lib.STRUCTS)) == -1


def test_ctypes_layout_matches_header():
    from glimpse_b200 import _lib

    names = ["gb_camera", "gb_image", "gb_surface", "gb_motion", "gb_plan", "gb_track_desc", "gb_stage_io"]
    prog = '#include <stdio.h>\n#include <stddef.h>\n#include "glimpse_b200.h"\nint main(void){\n'
    for n in names:
        prog += f'printf("{n} %zu\\n", sizeof({n}));\n'
    prog += 'printf("desc.plan %zu\\n", offsetof(gb_track_desc, plan));\n'
    prog += 'printf("desc.means %zu\\n", offsetof(gb_track_desc, means));\n'
    prog += 'printf("desc.seed %zu\\n", offsetof(gb_track_desc, seed));\n'
    prog += 'printf("image.cam %zu\\n", offsetof(gb_image, cam));\nreturn 0;}\n'
    with tempfile.TemporaryDirectory() as tmp:
        src, exe = os.path.join(tmp, "s.c"), os.path.join(tmp, "s")
        open(src, "w").write(prog)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        out = dict(line.split() for line in subprocess.check_output([exe], text=True).splitlines())
    for n in names:
        assert int(out[n]) == C.sizeof(getattr(_lib, n)), n
    assert int(out["desc.plan"]) == _lib.gb_track_desc.plan.offset
    assert int(out["desc.means"]) == _lib.gb_track_desc.means.offset
    assert int(out["desc.seed"]) == _lib.gb_track_desc.seed.offset
    assert int(out["image.cam"]) == _lib.gb_image.cam.offset


def test_camera_from_vector_matches_numpy_rotation():
    from glimpse_b200 import _lib, camera, synthetic

    lib = _lib.load()
    vec = synthetic.camera_vector(imgsz=(4288, 2848), f=(3700, 3690), c=(12.5, -8.25), xyz=(4.99e5, 6.77e6, 500.0),
                                  viewdir=(60.0, -25.0, 1.5), k=synthetic.FULL_K, p=synthetic.FULL_P)
    out = _lib.gb_camera()
    corr = np.array([6.3781e6, 0.13])
    assert lib.gb_camera_from_vector(vec.ctypes.data, corr.ctypes.data, C.byref(out)) == 0
    np.testing.assert_allclose(np.array(out.R[:]).reshape(3, 3), camera.rotation_matrix(vec[3:6]), atol=1e-15)
    assert list(out.imgsz[:]) == [4288, 2848]
    np.testing.assert_allclose(out.cc[:], [2144 + 12.5, 1424 - 8.25])
    assert out.has_corr == 1 and out.corr_c1 == 0.13 - 1 and out.corr_c2 == 2 * 6.3781e6


def test_plan_sizes():
    from glimpse_b200 import _lib

    lib = _lib.load()
    plan = _lib.gb_plan()
    S = _lib.GB_MODE_STREAM
    assert lib.gb_step_plan(1000, 15, 15, 10, 1, 0, S, C.byref(plan)) == 0
    assert plan.stream_nblk == 2 and plan.stream_block == 500 and plan.n_local == 1000 and plan.mode == S
    assert lib.gb_step_plan(10000, 15, 15, 1000, 1, 0, S, C.byref(plan)) == 0
    # particles of a point in equal even blocks of <= 768 (k_s4p's shared memory), 4 batches of points on 4 streams
    assert plan.stream_nblk == 14 and plan.stream_block == 716 and plan.stream_batch == 250 and plan.stream_slots == 4
    assert plan.surf_bytes > 700 * 1024 and plan.scratch_bytes > 1000 * (2 * 48 + 16 + 8) * 10000 + 1000 * plan.surf_bytes
    assert lib.gb_step_plan(100000, 31, 31, 1000, 1, 0, S, C.byref(plan)) == 0
    assert plan.stream_nblk == 131 and plan.stream_block * plan.stream_nblk >= 100000 and plan.stream_block % 2 == 0
    assert lib.gb_step_plan(1000, 40, 40, 10, 1, 0, S, C.byref(plan)) == -3  # template > 1024 px
    assert lib.gb_step_plan(1000, 15, 15, 10, 1, 0, 0, C.byref(plan)) == -1    # mode 0: round 1's cluster-per-point kernel, removed
    assert b"removed" in lib.gb_last_error()


def test_track_entry_points_refuse_frames_without_1_to_8_bands():
    """gb_track, gb_track_step and gb_track_init check every frame a time references for 1-8 bands before any device work
    (the tile kernels size their grey-level histograms for 255 * 8 + 1 levels); frames no time references are not read."""
    from glimpse_b200 import _lib

    lib = _lib.load()
    d = _lib.gb_track_desc()
    d.P, d.N, d.T, d.O, d.tile_w, d.tile_h = 1, 4, 2, 1, 15, 15
    assert lib.gb_step_plan(4, 15, 15, 1, 1, 0, _lib.GB_MODE_STREAM, C.byref(d.plan)) == 0
    fake = 1 << 20  # device pointers are not dereferenced by the argument checks
    for name in ("images", "mask", "first", "last", "motion", "surfaces", "state_a", "state_b", "means", "sigmas", "status",
                 "status_time", "obs_flags", "tmpl_tile", "tmpl_values", "tmpl_quantiles", "tmpl_nvalues", "tmpl_box", "tmpl_duv",
                 "scratch", "init_normals", "step_normals", "uniforms"):
        setattr(d, name, fake)
    images = (_lib.gb_image * 2)()
    offsets = np.array([0, 2], dtype=np.int32)
    index = np.zeros((2, 1), dtype=np.int32)  # image 1 is never referenced
    d.images_host, d.image_offset_host, d.image_index_host = C.addressof(images), offsets.ctypes.data, index.ctypes.data
    calls = {"gb_track": lambda: lib.gb_track(C.byref(d), None, None),
             "gb_track_step": lambda: lib.gb_track_step(C.byref(d), 1, None, None),
             "gb_track_init": lambda: lib.gb_track_init(C.byref(d), 0, None)}
    for name, call in calls.items():
        for nchan in (0, 9, -1, 255):
            images[0].nchan, images[1].nchan = nchan, 1
            assert call() == -1, (name, nchan)
            assert b"1 to 8 bands" in lib.gb_last_error(), (name, nchan)
        # 1-8 bands pass this check (the next one, a missing buffer, fails instead), whatever an unreferenced frame holds
        d.means = None
        for nchan in (1, 5, 8):
            images[0].nchan, images[1].nchan = nchan, 0
            assert call() == -1, (name, nchan)
            assert b"missing required buffer" in lib.gb_last_error(), (name, nchan)
        d.means = fake


def test_point_span_and_shards():
    from glimpse_b200.session import point_span
    from glimpse_b200.tracker import shard_bounds

    index = np.array([[-1, -1], [0, -1], [1, 0], [-1, 1], [-1, -1]])
    mask = np.array([[True, True], [True, False], [False, True], [False, False]])
    first, last = point_span(index, mask)
    np.testing.assert_array_equal(first, [1, 1, 2, 0])
    np.testing.assert_array_equal(last, [3, 2, 3, 4])  # no image at all: argmax semantics of the reference
    blocks = [shard_bounds(10, 4, r) for r in range(4)]
    assert blocks == [(0, 3), (3, 6), (6, 9), (9, 10)]
    assert [shard_bounds(2, 4, r) for r in range(4)] == [(0, 1), (1, 2), (2, 2), (2, 2)]


def _observers(n_frames=4, offset_days=0):
    import glimpse_b200 as gb

    t0 = datetime.datetime(2020, 1, 1) + datetime.timedelta(days=offset_days)
    images = []
    for i in range(n_frames):
        img = gb.Image(f"f{i}", cam=gb.Camera(imgsz=(20, 10), f=10), datetime=t0 + datetime.timedelta(days=i))
        img.array = np.zeros((10, 20), dtype=np.uint8)
        images.append(img)
    return gb.Observer(images)


def test_datetime_matching_follows_reference():
    import glimpse_b200 as gb

    a, b = _observers(4), _observers(3, offset_days=2)
    tracker = gb.Tracker([a, b])
    assert len(tracker.datetimes) == 5
    m = tracker.match_datetimes(tracker.datetimes)
    assert [v for v in m[:, 0]] == [0, 1, 2, 3, None]
    assert [v for v in m[:, 1]] == [None, None, 0, 1, 2]
    t0 = datetime.datetime(2020, 1, 1)
    with pytest.raises(ValueError, match="monotonic"):
        tracker.parse_datetimes([t0, t0 + datetime.timedelta(days=2), t0 + datetime.timedelta(days=1)])
    with pytest.raises(ValueError, match="Fewer than two"):
        tracker.parse_datetimes([t0 + datetime.timedelta(days=40), t0 + datetime.timedelta(days=41)])
    with pytest.warns(UserWarning, match="duplicate"):
        out = tracker.parse_datetimes([t0, t0, t0 + datetime.timedelta(days=1)])
    assert len(out) == 2
    back = tracker.parse_datetimes(tracker.datetimes[::-1])  # backward tracking is legal
    assert back[0] > back[-1]


def test_observer_validation_and_tile_box():
    import glimpse_b200 as gb

    obs = _observers(3)
    with pytest.raises(ValueError, match="two or greater"):
        gb.Observer(obs.images[:1])
    with pytest.raises(ValueError, match="stricly increasing"):
        gb.Observer(obs.images[::-1])
    np.testing.assert_array_equal(obs.tile_box((10.2, 5.4), (4, 4), img=0), [8, 3, 12, 7])
    with pytest.raises(IndexError):
        obs.tile_box((1.0, 5.0), (4, 4), img=0)
    assert obs.index(obs.images[1]) == 1 and obs.index(obs.datetimes[2]) == 2


def test_unsupported_options_raise_instead_of_falling_back():
    import glimpse_b200 as gb

    obs = _observers(3)
    day = datetime.timedelta(days=1)
    models = [gb.CartesianMotion(xy=(0, 0), time_unit=day, dem=0.0, n=10)]
    for kw in (dict(highpass={"size": 33}), dict(interpolation={"kx": 3, "ky": 3, "s": 1.0})):
        with pytest.raises(NotImplementedError):
            gb.Tracker([obs], **kw).track(models)
    with pytest.raises(ValueError, match="equal time units"):
        gb.Tracker([obs]).track(models + [gb.CartesianMotion(xy=(0, 0), time_unit=2 * day, dem=0.0, n=10)])

    from glimpse_b200.tracker import highpass_size, interpolation_degrees

    assert interpolation_degrees({}) == (3, 3) and interpolation_degrees({"kx": 1}) == (1, 3) and interpolation_degrees({"kx": 2, "ky": 5}) == (2, 5)
    with pytest.raises(ValueError, match="must be in"):
        interpolation_degrees({"kx": 6})

    assert highpass_size({"size": (3, 7)}) == (3, 7)  # (rows, columns), as scipy.ndimage.median_filter reads it
    assert highpass_size({"size": 4, "mode": "reflect", "origin": 0}) == (4, 4)
    from glimpse_b200 import _lib
    from glimpse_b200.tracker import highpass_params

    assert highpass_params({"size": (3, 5), "mode": "constant", "cval": 0.1, "origin": (1, -2)}) == (3, 5, _lib.GB_HP_MODES["constant"], 1, -2, 0.1, None)
    cross = np.array([[0, 1, 0], [1, 1, 1], [0, 1, 0]])
    assert highpass_params({"footprint": cross, "size": 9})[:2] == (3, 3) and highpass_params({"footprint": cross})[6] == [2, 7, 2]
    assert highpass_params({"footprint": np.ones((3, 7))})[6] is None  # a full footprint is a size
    assert highpass_params({"size": 5, "mode": "grid-wrap"})[2] == _lib.GB_HP_MODES["wrap"]
    with pytest.raises(ValueError, match="invalid origin"):  # scipy: -(size // 2) <= origin <= (size - 1) // 2
        highpass_params({"size": 4, "origin": 2})
    with pytest.raises(RuntimeError, match="boundary mode not supported"):
        highpass_params({"size": 5, "mode": "periodic"})

    class Custom:
        n, time_unit = 10, day

    from glimpse_b200.session import adopt_model

    with pytest.raises(NotImplementedError, match="no device kernel"):
        adopt_model(Custom())


def test_no_cpu_fallback_without_cuda():
    import torch

    import glimpse_b200 as gb

    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    cam = gb.Camera(imgsz=10, f=10)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        cam.xyz_to_uv(np.zeros((1, 3)))
    obs = _observers(3)
    models = [gb.CartesianMotion(xy=(0, 0), time_unit=datetime.timedelta(days=1), dem=0.0, n=10)] * 2
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        gb.Tracker([obs]).track(models)


WORKER = r"""
import os, sys, datetime
import numpy as np
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, os.path.join(sys.argv[1], "tests"))
import torch, torch.distributed as dist
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%s" % sys.argv[2], rank=int(sys.argv[3]), world_size=2)
import glimpse_b200 as gb
from test_host import _observers
obs = _observers(4)
day = datetime.timedelta(days=1)
models = [gb.CartesianMotion(xy=(float(i), 0), time_unit=day, dem=0.0, n=8) for i in range(5)]
tracker = gb.Tracker([obs])
seen = {}
def fake_local(models, image_index, taus, tile_size, mask, cov, parts, point_offset=0, dist=None, seed=None, n_particles=0, gather=None):
    # stands in for the GPU compute: encodes (global point index, time) so the gather can be checked
    from glimpse_b200.session import empty_result
    P, T, O = len(models), image_index.shape[0], image_index.shape[1]
    out = empty_result(P, T, O, cov, parts, N=8)
    for i, m in enumerate(models):
        out["means"][i] = m.xy[0] * 100 + np.arange(T)[:, None]
        out["sigmas"][i] = point_offset + i
    if P:
        out["status"][-1] = 5 if point_offset == 0 else 0
        out["status_time"][-1] = 2
    seen["block"] = (point_offset, P)
    return out
tracker._track_local = fake_local
tracks = tracker.track(models)
assert seen["block"] == ((0, 3) if dist.get_rank() == 0 else (3, 2)), seen
assert tracks.means.shape == (5, 4, 6)
for i in range(5):
    assert np.all(tracks.means[i] == i * 100 + np.arange(4)[:, None]) and np.all(tracks.sigmas[i] == i)
assert isinstance(tracks.errors[2], IndexError) and all(tracks.errors[i] is None for i in (0, 1, 3, 4))
# three points on two ranks with the particles returned: rank 1 holds one point; then one point: rank 1 is idle and
# contributes blocks of zero rows with the right particle count (shapes must agree across ranks)
for n in (3, 1):
    seen.clear()
    tracks = tracker.track(models[:n] if n > 1 else models[:1] * 1, return_particles=True) if n > 1 else None
    if n > 1:
        assert tracks.particles.shape == (3, 4, 8, 6) and tracks.weights.shape == (3, 4, 8)
        assert seen["block"] == ((0, 2) if dist.get_rank() == 0 else (2, 1)), seen
# points that outgrew their search windows: every rank runs its own again, only the patched rows are gathered
from glimpse_b200 import _lib
from glimpse_b200.session import empty_result
def failing_local(models, image_index, *a, point_offset=0, **kw):
    out = fake_local(models, image_index, *a, point_offset=point_offset, **kw)
    out["status"][:] = 0
    for i in range(len(models)):
        if point_offset + i in (1, 3, 4):
            out["status"][i], out["means"][i] = _lib.GB_ST_WINDOW_TOO_LARGE, np.nan
    return out
def fake_rows(failed, seed, models, image_index, *a):
    point_offset = a[-1]
    if len(failed) == 0:
        return None
    rows = empty_result(len(failed), image_index.shape[0], image_index.shape[1], False, False)
    for j, i in enumerate(failed):
        rows["means"][j] = 1000 + point_offset + i
        rows["sigmas"][j] = 7
    return rows
tracker._track_local, tracker._rerun_rows = failing_local, fake_rows
tracks = tracker.track(models)
assert all(e is None for e in tracks.errors), tracks.errors
assert [float(tracks.means[i, 0, 0]) for i in range(5)] == [0.0, 1001.0, 200.0, 1003.0, 1004.0], tracks.means[:, 0, 0]
assert np.all(tracks.sigmas[[1, 3, 4]] == 7)
tracker._track_local = fake_local
local = fake_local(models[:1] if dist.get_rank() == 0 else [], np.zeros((4, 1), dtype=np.int32), None, None, None, False, True,
                   point_offset=dist.get_rank(), n_particles=8)
merged = gb.Tracker._gather(dist, local, 1, 2)
assert merged["particles"].shape == (1, 4, 8, 6) and merged["means"].shape == (1, 4, 6) and merged["status"].shape == (1,)
dist.barrier(); dist.destroy_process_group()
print("rank", sys.argv[3], "ok")
"""


def test_points_shard_across_ranks_and_gather_over_gloo():
    """world_size 2 on CPU: contiguous blocks of points per rank, one final all-gather, every rank
    returns the full Tracks (the compute itself is stubbed: it has no CPU path)."""
    import socket

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    procs = [subprocess.Popen([sys.executable, "-c", WORKER, ROOT, str(port), str(r)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    for r, (p, out) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, out
        assert f"rank {r} ok" in out


def test_tracks_from_multiple_and_average_match_the_reference():
    """Tracks.from_multiple / Tracks.average (reference tracks.py:151-203, helpers.sum_normals) against vectors produced
    by the unmodified reference (tests/golden/make_tracks_golden.py), with missing values in one or both runs."""
    import glimpse_b200 as gb

    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "tracks_merge.npz"))
    day = datetime.timedelta(days=1)
    dts = [datetime.datetime(2020, 1, 1) + i * day for i in range(g["m1"].shape[1])]
    a = gb.Tracks(datetimes=dts, time_unit=day, means=g["m1"], sigmas=g["s1"])
    b = gb.Tracks(datetimes=dts, time_unit=day, means=g["m2"], sigmas=g["s2"])
    for ign in (0, 1):
        merged = gb.Tracks.from_multiple([a, b], ignore_nan=bool(ign))
        np.testing.assert_allclose(merged.means, g[f"merged_means_{ign}"], rtol=1e-13, atol=0, equal_nan=True)
        np.testing.assert_allclose(merged.sigmas, g[f"merged_sigmas_{ign}"], rtol=1e-13, atol=0, equal_nan=True)
        am, asg = a.average(ignore_nan=bool(ign))
        np.testing.assert_allclose(am, g[f"avg_means_{ign}"], rtol=1e-13, atol=0, equal_nan=True)
        np.testing.assert_allclose(asg, g[f"avg_sigmas_{ign}"], rtol=1e-12, atol=0, equal_nan=True)
    with pytest.raises(ValueError, match="Datetimes are not equal"):
        gb.Tracks.from_multiple([a, gb.Tracks(datetimes=dts[::-1], time_unit=day, means=g["m2"], sigmas=g["s2"])])
    with pytest.raises(ValueError, match="Time units are not equal"):
        gb.Tracks.from_multiple([a, gb.Tracks(datetimes=dts, time_unit=2 * day, means=g["m2"], sigmas=g["s2"])])


def test_points_are_blocked_by_device_memory():
    """BASELINE.json config 5 (100 000 points x 10 000 particles x 365 frames) needs ~300 GB of work buffers: more than one
    B200 has, so a one- or two-GPU run advances consecutive blocks of points; 12 500 points (one of eight ranks) fit."""
    from glimpse_b200 import _lib, build
    from glimpse_b200.session import points_per_session, session_bytes

    build.build()
    lib = _lib.load()
    frames = ([], None)  # no frame to read: the plan of uint8 frames
    shape = dict(N=10000, T=365, O=1, tw=15, th=15, return_covariances=False, return_particles=False)
    whole = session_bytes(lib, *frames, 100000, **shape)
    assert 250e9 < whole < 350e9
    assert session_bytes(lib, *frames, 12500, **shape) < 45e9
    block = points_per_session(lib, *frames, 100000, int(160e9), **shape)
    assert 45000 < block < 65000
    assert session_bytes(lib, *frames, block, **shape) <= 160e9 < session_bytes(lib, *frames, block + 1, **shape)
    assert points_per_session(lib, *frames, 1000, int(160e9), **shape) == 1000
    assert points_per_session(lib, *frames, 1000, 1, **shape) == 1  # never less than one point


def test_session_bytes_plan_ranked_frames_as_the_session_does():
    """A uint16 observer makes Session plan ranked frames, whose surface regions hold a rank histogram of the largest window
    (twice the bytes at 15 x 15 and 10 000 particles).  session_bytes plans the same, so the blocks Tracker cuts a large
    track into fit the device."""
    from glimpse_b200 import _lib
    from glimpse_b200.session import session_bytes

    lib = _lib.load()
    P, N, T, O, tw, th = 1000, 10000, 4, 2, 15, 15
    observers = [_observers(T), _observers(T)]
    index = np.array([[0, 0], [1, -1], [2, 1], [3, 2]])
    shape = dict(N=N, T=T, O=O, tw=tw, th=th, return_covariances=False, return_particles=False)
    uint8 = session_bytes(lib, observers, index, P, **shape)
    for image in observers[1].images:
        image.array = np.zeros((10, 20), dtype=np.uint16)
    uint16 = session_bytes(lib, observers, index, P, **shape)
    plans = {}
    for flags in (0, _lib.GB_PLAN_RANKED_FRAMES):
        plans[flags] = _lib.gb_plan()
        assert lib.gb_step_plan_ex(N, tw, th, P, O, flags, _lib.GB_MODE_STREAM, _lib.GB_WINDOW_MARGIN, C.byref(plans[flags])) == 0
    ranked = plans[_lib.GB_PLAN_RANKED_FRAMES]
    # per point: particle states and weights, three template arrays and 40 B of template scalars per observer, moments and
    # sigmas, flag bytes and window sizes per time and observer, status
    per_point = 2 * 48 * N + 8 * N + O * (3 * tw * th * 8 + 40) + T * 12 * 8 + T * O * 9 + 16
    assert uint16 == ranked.scratch_bytes + P * per_point
    assert ranked.surf_bytes > plans[0].surf_bytes
    assert uint16 - uint8 == P * O * (ranked.surf_bytes - plans[0].surf_bytes)


def test_blocks_and_second_runs_are_assembled_on_the_host(monkeypatch):
    """Host logic of Tracker._track_local with the device session stubbed (it has no CPU path): consecutive blocks of
    points, the second run of points that outgrew the window capacity (same Philox key, own global index, largest
    capacity), and what is reported in Tracker.last_run."""
    import glimpse_b200 as gb
    from glimpse_b200 import _lib, session as session_mod

    created = []

    class FakeSession:
        def __init__(self, tracker, models, image_index, taus, tile_size, observer_mask, return_covariances=False,
                     return_particles=False, point_offset=0, draws=None, dist=None, window_margin=None, seed=None):
            self.models, self.offset, self.margin = models, point_offset, window_margin
            self.T, self.O = image_index.shape
            self.seed_used = 4242 if seed is None else seed
            assert len(observer_mask) == len(models)
            created.append(self)

        def run(self):
            pass

        def fetch(self):
            P = len(self.models)
            out = session_mod.empty_result(P, self.T, self.O, False, False)
            for i, m in enumerate(self.models):
                g = self.offset + i
                out["means"][i] = g
                # global points 1 and 4 outgrow the default window capacity; the second run (largest capacity) succeeds
                if g in (1, 4) and self.margin is None:
                    out["status"][i], out["status_time"][i] = _lib.GB_ST_WINDOW_TOO_LARGE, 2
                    out["means"][i] = np.nan
            self.stats = {"plan": {}, "kernel_launches": 10, "h2d_bytes": 100, "d2h_bytes": 7,
                          "window_width": np.arange(P), "window_height": np.arange(P)}
            return out

        def final_state(self):
            return "particles", "weights", self.offset

    monkeypatch.setattr(session_mod, "Session", FakeSession)
    obs = _observers(4)
    day = datetime.timedelta(days=1)
    models = [gb.CartesianMotion(xy=(float(i), 0), time_unit=day, dem=0.0, n=8) for i in range(5)]
    tracker = gb.Tracker([obs])
    tracker._points_per_session = lambda *a, **k: 2
    tracks = tracker.track(models)
    blocks = [(s.offset, len(s.models), s.margin) for s in created]
    # blocks of 2, 2, 1 points; then points 1 and 4 are run again
    assert blocks == [(0, 2, None), (2, 2, None), (4, 1, None), (1, 1, _lib.GB_WINDOW_MARGIN_MAX), (4, 1, _lib.GB_WINDOW_MARGIN_MAX)]
    assert len({s.seed_used for s in created}) == 1 and created[0].seed_used != 4242  # one key per track() call, drawn by the Tracker
    assert all(e is None for e in tracks.errors)
    np.testing.assert_array_equal(tracks.means[:, 0, 0], np.arange(5.0))
    assert tracker.last_run["sessions"] == 3 and tracker.last_run["kernel_launches"] == 30
    assert len(tracker.last_run["window_width"]) == 5 and tracker._rerun_points == [1, 4]
    assert tracker.templates == 4  # the state the last block left, as the reference keeps the last track's
    # the reference's draw sequence cannot be replayed: the error stays
    created.clear()
    tracker = gb.Tracker([obs], rng="numpy")
    tracker._points_per_session = lambda *a, **k: 5
    tracks = tracker.track(models)
    assert [isinstance(e, MemoryError) for e in tracks.errors] == [False, True, False, False, True]
    assert len(created) == 1


def test_observer_subset_split_and_select_datetimes():
    """Observer.subset / split (reference observer.py:455-493) and helpers.select_datetimes / datetime_range with the known
    answers of the reference's doctests (helpers.py:1870-1922)."""
    import glimpse_b200 as gb
    from glimpse_b200.observer import datetime_range, select_datetimes

    t = [datetime.datetime(2020, 1, 1, 0, 0, x) for x in (0, 1, 2, 4, 5)]
    assert select_datetimes(t).tolist() == [True] * 5
    assert select_datetimes(t, start=t[1]).tolist() == [False, True, True, True, True]
    assert select_datetimes(t, start=t[1], end=t[1]).tolist() == [False, True, False, False, False]
    snap = datetime.timedelta(seconds=2)
    assert select_datetimes(t, snap=snap).tolist() == [True, False, True, True, True]
    assert select_datetimes(t, snap=snap, maxdt=0 * snap).tolist() == [True, False, True, True, False]
    with pytest.raises(ValueError, match="Start datetime is after end datetime"):
        select_datetimes(t, start=t[3], end=t[1])
    base = (2020, 1, 1, 0, 0)
    rng = datetime_range(datetime.datetime(*base, 0), datetime.datetime(*base, 2), datetime.timedelta(seconds=1))
    assert list(rng) == [datetime.datetime(*base, s) for s in (0, 1, 2)]
    obs = _observers(9)
    sub = obs.subset(start=obs.datetimes[2], end=obs.datetimes[5])
    assert [img is obs.images[2 + i] for i, img in enumerate(sub.images)] == [True] * 4 and sub.sigma == obs.sigma
    parts = obs.split(2)  # two halves sharing one image (overlap = 1)
    assert [len(p.images) for p in parts] == [5, 5] and parts[1].images[0] is parts[0].images[-1]
    parts = obs.split(2, overlap=0)
    assert [len(p.images) for p in parts] == [5, 4] and parts[1].images[0] is obs.images[5]
    parts = obs.split([obs.datetimes[3]], overlap=2)
    assert [len(p.images) for p in parts] == [4, 7] and parts[1].images[0] is obs.images[2]
    with pytest.raises(ValueError, match="Shift larger than 0.5 pixels"):
        obs.shift_tile(np.zeros((5, 5)), (0.6, 0.0))
    with pytest.raises(NotImplementedError):
        obs.sample_tile(np.zeros((1, 2)), np.zeros((5, 5)), (0, 0, 5, 5), kx=6)


def _reference_results(lower, scene):
    """``lower(scene, api)`` with the unmodified reference (``oracle/ref_shim.py``), or None where it cannot be imported."""
    from oracle import ref_shim

    return lower(scene, ref_shim.import_reference()) if ref_shim.available() else None


@pytest.mark.parametrize("kind", ["cartesian", "cylindrical", "tangent_cartesian", "tangent_cylindrical"])
def test_reference_objects_lower_to_the_same_tables(kind):
    """INTEGRATION.md §1: the reference's own Observer / Image / Camera / motion-model / Raster objects are accepted as they
    are.  Built from one scene, this package's objects lower to the gb_camera / gb_motion / gb_surface tables (host side of
    the C ABI) stored in tests/golden/lowering.npz, including gridded DEMs, a viewshed raster and cameras with curvature /
    refraction corrections; where the reference can be imported, its objects must lower to byte-identical tables."""
    import helpers

    import glimpse_b200 as gb

    scene = helpers.lowering_scene(kind)
    mine = helpers.lowered_tables(scene, gb)
    golden = helpers.load_golden("lowering")
    helpers.assert_tables_close(mine, {k.split(".", 1)[1]: golden[k] for k in golden.files if k.split(".", 1)[0] == kind})
    assert len(mine["surfaces"]) >= (3 if kind.startswith("tangent") else 2)
    theirs = _reference_results(helpers.lowered_tables, scene)
    if theirs is not None:
        assert sorted(theirs) == sorted(mine)
        for key in mine:
            np.testing.assert_array_equal(theirs[key], mine[key], err_msg=key)


def test_reference_raster_frames_lower_to_the_same_affine_camera():
    """An Observer of orthoimages: this package's Raster frames lower to the affine gb_camera and answer xyz_to_uv /
    uv_to_xyz / inbounds / read / d / size (raster.py:119-122, 339-341, 423-459, 763-836) as stored in
    tests/golden/lowering.npz; where the reference can be imported, its Raster frames must give exactly the same."""
    import helpers
    from glimpse_b200 import synthetic
    from glimpse_b200.session import lower_grid_camera

    import glimpse_b200 as gb

    scene = helpers.raster_frames_scene()
    mine = helpers.raster_frame_results(scene, gb)
    golden = helpers.load_golden("lowering")
    helpers.assert_tables_close(mine, {k.split(".", 1)[1]: golden[k] for k in golden.files if k.split(".", 1)[0] == "raster"})
    theirs = _reference_results(helpers.raster_frame_results, scene)
    if theirs is not None:
        for key in mine:
            np.testing.assert_array_equal(theirs[key], mine[key], err_msg=key)
    for b in synthetic.build(scene, gb)[0][0].images:
        cb = lower_grid_camera(b)
        assert cb.affine == 1 and tuple(cb.imgsz) == (320, 240)
        assert cb.f[0] > 0 > cb.f[1]  # north-up: y decreases with the row
        assert b.read().dtype == np.uint8
        with pytest.raises(ValueError):
            b.read(box=(-1, 0, 5, 5))
        with pytest.raises(ValueError):
            b.read(box=(0.5, 0, 5, 5))
    with pytest.raises(NotImplementedError):
        lower_grid_camera(object())


def test_frames_of_other_types_are_accepted_as_numpy_would_promote_them():
    """tracker.py:522-526 takes frames of any dtype: uint8 keeps the integer tile pipeline, uint16 / float32 / float64 go to the
    device as they are (rank pipeline), other integer types as float64 (exact), float16 as float32."""
    from glimpse_b200 import _lib
    from glimpse_b200.session import device_frame, frames_need_ranks

    for dtype, want in ((np.uint8, "uint8"), (np.uint16, "uint16"), (np.float32, "float32"), (np.float64, "float64"), (np.int16, "float64"),
                        (np.int32, "float64"), (np.uint32, "float64"), (np.bool_, "float64"), (np.float16, "float32")):
        out = device_frame(np.ones((4, 6, 3), dtype=dtype)[:, ::2])  # (a non-contiguous view is copied)
        assert out.dtype.name == want and out.flags.c_contiguous and out.shape == (4, 3, 3) and want in _lib.GB_PIX
    with pytest.raises(NotImplementedError):
        device_frame(np.ones((4, 6), dtype=complex))
    with pytest.raises(NotImplementedError):
        device_frame(np.ones((4, 6, 9), dtype=np.uint8))
    obs = _observers(3)
    index = np.array([[0], [1], [2]])
    assert not frames_need_ranks([obs], index)
    obs.images[1].array = np.zeros((10, 20), dtype=np.uint16)
    assert frames_need_ranks([obs], index) and not frames_need_ranks([obs], np.array([[0], [-1], [2]]))
