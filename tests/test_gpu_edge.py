"""Edge cases and size-independent properties of the device Tracker, checked against the oracle
(free-running with the reference's draw order) or against invariants of the algorithm."""
import datetime
import warnings

import numpy as np
import pytest

import helpers
import scenes
from glimpse_b200 import synthetic
from oracle import tracker_oracle as orc

pytestmark = pytest.mark.gpu
MODES = ["stream"]


def run_both(scene, seed, mode, points=None, viewshed=None, oracle_viewshed=None, exact=True, **track_kw):
    import glimpse_b200 as gb

    observers, models = synthetic.build(scene, gb, points=points)
    tracker = gb.Tracker(observers, viewshed=viewshed, rng="numpy", mode=mode)
    np.random.seed(seed)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        tracks = tracker.track(models, tile_size=scene.tile_size, **track_kw)
    obs, specs, taus, index = helpers.oracle_inputs(scene, points=points)
    np.random.seed(seed)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref = orc.track(obs, specs, taus, index, tile_size=scene.tile_size, viewshed=oracle_viewshed, exact=exact,
                        return_covariances=track_kw.get("return_covariances", False),
                        return_particles=track_kw.get("return_particles", False),
                        observer_mask=track_kw.get("observer_mask"))
    return tracks, ref, tracker


def assert_close_to_oracle(tracks, ref, sig_tol=1e-5):
    """Free-running agreement of the means in units of the reference's sigma.  The default asks for identical ancestors
    everywhere (achieved: <= 1e-7 sigma); tests with thousands of particles per point, where one flipped ancestor turns the
    rest of the track into another realisation of the filter (tests/test_gpu_track.py), pass their own bound."""
    sig = ref.sigmas if ref.sigmas.ndim == 3 else np.sqrt(np.einsum("ptii->pti", ref.sigmas))
    both = ~np.isnan(ref.means[..., 0])
    assert np.array_equal(~np.isnan(tracks.means[..., 0]), both)
    d = np.abs(tracks.means - ref.means) / np.maximum(sig, 1e-9)
    worst = float(np.nanmax(d[..., [0, 1, 3, 4]]))
    assert worst < sig_tol, f"max |dmean| = {worst:.3g} sigma"



@pytest.mark.parametrize("mode", MODES)
def test_template_beyond_image_is_an_index_error(cuda, mode):
    """raster.py:417-418 via observer.py:115-130: captured per track with >= 2 tracks, raised with one."""
    import glimpse_b200 as gb

    scene = synthetic.nadir_scene(seed=4, n_points=3, n_particles=256, n_frames=4, imgsz=(320, 240), margin_px=90)
    # (the failing track goes last: a track that stops early leaves its later draws unconsumed in the reference,
    #  so tracks after it see a shifted random stream)
    scene.points[2, 0] = (320 / 2 - 3) * 0.2  # 3 px from the right edge: the 15 x 15 template does not fit
    tracks, ref, _ = run_both(scene, 11, mode)
    assert [type(e).__name__ if e else None for e in tracks.errors] == [None, None, "IndexError"]
    assert isinstance(ref.errors[2], IndexError)
    assert np.isnan(tracks.means[2]).all() and not np.isnan(tracks.means[:2]).any()
    assert_close_to_oracle(tracks, ref)
    observers, models = synthetic.build(scene, gb, points=[2])
    with pytest.raises(IndexError, match="Box extends beyond grid bounds"):
        gb.Tracker(observers, rng="numpy", mode=mode).track(models, tile_size=scene.tile_size)


@pytest.mark.parametrize("mode", MODES)
def test_particles_leaving_the_frame_skip_the_image_with_a_warning(cuda, mode):
    """tracker.py:597-601: the observer contributes nothing, the filter keeps running on the motion model."""
    scene = synthetic.nadir_scene(seed=6, n_points=2, n_particles=256, n_frames=6, imgsz=(320, 240), margin_px=100,
                                  velocity_sigma=0.3)
    scene.points[0, 0] = (320 / 2 - 24) * 0.2  # template fits, the growing cloud does not
    scene.motion["vxyz"] = (2.0, 0.0, 0.0)      # 10 px / day towards the edge
    tracks, ref, _ = run_both(scene, 21, mode)
    assert tracks.errors[0] is None and tracks.warnings[0] is not None
    assert all("too close to or beyond image bounds" in str(w) for w in tracks.warnings[0])
    assert (ref.skipped[0] == 2).sum() == len(tracks.warnings[0]) > 0
    assert_close_to_oracle(tracks, ref)


@pytest.mark.parametrize("mode", MODES)
def test_viewshed_and_gridded_dem(cuda, mode):
    """tracker.py:114-117 (nearest viewshed sample) and motion.py:181-204 with a 2-D DEM / DEM sigma
    (bilinear Raster.sample, raster.py:891-1027)."""
    import glimpse_b200 as gb

    scene = synthetic.nadir_scene(seed=8, n_points=3, n_particles=300, n_frames=5, imgsz=(320, 240), margin_px=90)
    rng = np.random.RandomState(0)
    dem = 0.5 * rng.rand(12, 16)
    sig = 0.5 + 0.1 * rng.rand(12, 16)
    x, y = (-40.0, 40.0), (30.0, -30.0)  # north-up raster: y decreasing
    scene.motion.update(dem=gb.Raster(dem, x=x, y=y), dem_sigma=gb.Raster(sig, x=x, y=y))
    scene.points = scene.points[[0, 2, 1]]  # the eastern point last (see the note on draw order above)
    vis = np.ones((12, 16))
    vis[:, 10:] = 0  # the eastern point (x = +14 m) starts on non-visible cells
    viewshed = gb.Raster(vis, x=x, y=y)
    observers, models = synthetic.build(scene, gb)
    scene.motion.update(dem=0.0, dem_sigma=0.0)  # placeholders for the oracle specs, replaced below
    tracker = gb.Tracker(observers, viewshed=viewshed, rng="numpy", mode=mode)
    np.random.seed(5)
    tracks = tracker.track(models, tile_size=scene.tile_size)
    obs, specs, taus, index = helpers.oracle_inputs(scene)
    for sp in specs:
        sp.dem, sp.dem_sigma = orc.Surface(dem, x, y), orc.Surface(sig, x, y)
    np.random.seed(5)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref = orc.track(obs, specs, taus, index, tile_size=scene.tile_size, viewshed=orc.Surface(vis, x, y), exact=True)
    kinds = [type(e).__name__ if e else None for e in tracks.errors]
    assert kinds == [type(e).__name__ if e else None for e in ref.errors]
    assert "ValueError" in kinds and None in kinds
    assert "non-visible viewshed" in str([e for e in tracks.errors if e][0])
    assert_close_to_oracle(tracks, ref)
    z_ok = ~np.isnan(ref.means[..., 2])
    assert np.max(np.abs(tracks.means[..., 2][z_ok] - ref.means[..., 2][z_ok])) < 0.05 * np.nanmax(ref.sigmas[..., 2])


@pytest.mark.parametrize("mode", MODES)
def test_cylindrical_zero_speed_gives_nan_error(cuda, mode):
    """motion.py:296-303: vr = 0 -> 0/0 -> 'Some particles have missing (NaN) values'."""
    scene = synthetic.nadir_scene(seed=3, n_points=2, n_particles=128, n_frames=4, imgsz=(320, 240), margin_px=100,
                                  kind="cylindrical")
    scene.motion.update(vrthz=(0.0, 0.0, 0.0), vrthz_sigma=(0.0, 0.0, 0.0))
    tracks, ref, _ = run_both(scene, 2, mode)
    assert all(isinstance(e, ValueError) and "NaN" in str(e) for e in tracks.errors)
    assert all(isinstance(e, ValueError) for e in ref.errors)
    assert not np.isnan(tracks.means[:, 0]).any() and np.isnan(tracks.means[:, 1:]).all()


@pytest.mark.parametrize("mode", MODES)
def test_large_template_many_particles_and_mask(cuda, mode):
    """config-4 shape shrunk (31 x 31 template, N = 20 000: scratch / multi-CTA paths), covariances,
    and an observer mask that removes the only observer for one point (motion-only track)."""
    scene = synthetic.nadir_scene(seed=12, n_points=3, n_particles=20000, n_frames=4, imgsz=(400, 300), margin_px=130,
                                  tile_size=(31, 31), velocity_sigma=0.5)
    mask = np.array([[True], [True], [False]])
    tracks, ref, tracker = run_both(scene, 9, mode, return_covariances=True, observer_mask=mask)
    assert all(e is None for e in tracks.errors)
    assert tracks.covariances.shape == (3, 4, 6, 6) and tracks.sigmas is None
    assert_close_to_oracle(tracks, ref, sig_tol=5e-3)  # 20 000 particles: one ancestor may flip (5e-4 sigma measured)
    c_ref, c = ref.sigmas, tracks.covariances
    scale = np.sqrt(np.einsum("ptii,ptjj->ptij", c_ref, c_ref))
    ok = scale > 0
    assert np.max(np.abs(c - c_ref)[ok] / scale[ok]) < 0.05
    # the unobserved point: weights stay uniform, positions follow the motion model only
    assert np.allclose(tracks.means[2, :, 3], scene.truth_velocity[0], atol=0.02)


@pytest.mark.parametrize("mode", MODES)
def test_backward_tracking_and_api_shapes(cuda, mode):
    """Decreasing datetimes are legal (tracker.py:446-450): negative time steps."""
    import glimpse_b200 as gb

    scene = synthetic.nadir_scene(seed=14, n_points=2, n_particles=400, n_frames=6, imgsz=(320, 240), margin_px=100)
    observers, models = synthetic.build(scene, gb)
    tracker = gb.Tracker(observers, seed=3, mode=mode)
    back = tracker.track(models, datetimes=tracker.datetimes[::-1], tile_size=scene.tile_size, return_particles=True)
    assert back.datetimes[0] > back.datetimes[-1]
    assert back.particles.shape == (2, 6, 400, 6) and back.weights.shape == (2, 6, 400)
    assert np.all(np.abs(back.vxyz[:, -1, 0] - scene.truth_velocity[0]) < 0.05)  # velocity keeps its sign, time runs backwards
    # reported moments are those of the returned (resampled) particles and weights (tracker.py:350-354)
    for p in range(2):
        for t in range(6):
            m = np.average(back.particles[p, t], weights=back.weights[p, t], axis=0)
            assert np.max(np.abs(m - back.means[p, t]) / np.maximum(np.abs(m), 1e-3)) < 1e-11
            s = np.sqrt(np.average((back.particles[p, t] - m) ** 2, weights=back.weights[p, t], axis=0))
            assert np.allclose(s, back.sigmas[p, t], rtol=1e-7, atol=1e-12)
    reduced = tracker.track(models, tile_size=scene.tile_size, reduce_particles=lambda ps, ws: ps.shape + ws.shape)
    assert reduced.particles is None and reduced.reduced == [(6, 400, 6, 6, 400)] * 2
    assert tracker.particles.shape == (400, 6) and tracker.templates[0]["tile"].shape == (15, 15)


@pytest.mark.parametrize("mode", MODES)
def test_resampling_properties_at_scale(cuda, mode):
    """Size-independent invariants of systematic resampling at N = 100 000 through the production kernel:
    uniform weights -> identity; any weights -> sorted ancestors with |count_i - N w_i / W| < 1."""
    import ctypes as C

    import glimpse_b200 as gb
    from glimpse_b200 import _lib
    from glimpse_b200.session import Session

    torch = cuda
    N, P = 100000, 3
    scene = synthetic.nadir_scene(seed=1, n_points=P, n_particles=N, n_frames=3, imgsz=(320, 240), margin_px=100)
    observers, models = synthetic.build(scene, gb)
    tracker = gb.Tracker(observers, seed=7, mode=mode)
    index = np.array([[0], [1], [2]], dtype=np.int32)
    s = Session(tracker, models, index, np.ones(2), scene.tile_size, np.ones((P, 1), dtype=bool))
    s.init(0)
    rng = np.random.RandomState(3)
    w = np.ones((P, N))
    w[1] = rng.rand(N) ** 6
    w[2] = 1e-300
    w[2, 77] = 1.0  # degenerate: one particle takes everything
    fw = torch.as_tensor(w).to(s.device)
    idx = torch.full((P, N), -1, dtype=torch.int32, device=s.device)
    io = _lib.gb_stage_io()
    io.force_weights, io.dump_indices = fw.data_ptr(), idx.data_ptr()
    s.step(1, io)
    torch.cuda.synchronize()
    assert (s.buf["status"].cpu().numpy() == 0).all()
    got = idx.cpu().numpy()
    np.testing.assert_array_equal(got[0], np.arange(N))
    assert np.all(np.diff(got[1]) >= 0) and got[1].min() >= 0 and got[1].max() < N
    counts = np.bincount(got[1], minlength=N)
    assert np.all(np.abs(counts - N * w[1] / w[1].sum()) < 1.0 + 1e-6)
    assert np.all(got[2] == 77)
    # the state written for the next step is the gathered one
    state = (s.buf["state_b"] if 1 & 1 else s.buf["state_a"]).cpu().numpy()
    assert np.all(state[2] == state[2][:, :1])


@pytest.mark.parametrize("n_particles", [1001, 37, 1537])
def test_odd_and_ragged_particle_counts(cuda, n_particles):
    """Particle counts that are odd, smaller than a warp-multiple, or leave a ragged last block: k_s4p takes its
    element-wise staging path instead of bulk copies (odd N), the last block of a point is shorter than the others."""
    scene = synthetic.nadir_scene(seed=21, n_points=3, n_particles=n_particles, n_frames=5, imgsz=(320, 240), margin_px=90)
    tracks, ref, _ = run_both(scene, 5, "stream", return_particles=True)
    assert all(e is None for e in tracks.errors)
    assert_close_to_oracle(tracks, ref, sig_tol=1e-3)
    # resampled particles are exact copies of the oracle's (same ancestors)
    same = np.isclose(tracks.particles, ref.particles, rtol=0, atol=1e-9).all(axis=3)
    assert same.mean() > 0.999


def test_three_observers_use_the_generic_observer_loop(cuda):
    """k_s4p unrolls its first two observers; a third one goes through the generic loop (shared-memory box atomics)."""
    import scenes

    scene = synthetic.nadir_scene(seed=23, n_points=2, n_particles=600, n_frames=5, imgsz=(320, 240), margin_px=100)
    scenes.add_second_observer(scene)
    first = scene.observers[0]
    # third station: the first one's frames under a slightly looser pixel sigma
    scene.observers.append(synthetic.ObserverScene([f.copy() for f in first.frames], first.cams.copy(), list(first.datetimes), sigma=0.5))
    tracks, ref, _ = run_both(scene, 9, "stream")
    assert_close_to_oracle(tracks, ref, sig_tol=1e-3)


def test_collapsed_weights_give_one_parent_many_children(cuda):
    """A tiny pixel sigma concentrates the weight on a few particles: one k_s4p block then owns far more children
    than parents (several chunks of its child loop) while the other blocks own none."""
    scene = synthetic.nadir_scene(seed=25, n_points=2, n_particles=3000, n_frames=4, imgsz=(320, 240), margin_px=100)
    scene.observers[0].sigma = 0.02  # (much smaller and every weight underflows to the 1e-300 floor: uniform again)
    tracks, ref, _ = run_both(scene, 13, "stream", return_particles=True)
    # 1 / (2 sigma^2) = 1250 amplifies the float32 rounding of the SSD surface (3e-7 relative) into weight differences
    # of ~4e-4, so a few ancestors may differ from the oracle's after several updates: looser bounds than elsewhere
    assert_close_to_oracle(tracks, ref, sig_tol=0.02)
    # the collapse really happened: after the first update all 3000 particles descend from < 100 parents
    uniq = [len(np.unique(tracks.particles[p, 1, :, 0])) for p in range(2)]
    assert max(uniq) < 100
    same = np.isclose(tracks.particles, ref.particles, rtol=0, atol=1e-9).all(axis=3)
    assert same[:, :2].mean() > 0.99 and same.mean() > 0.95, (same[:, :2].mean(), same.mean())


def test_tangent_model_keeps_its_weights_when_no_image_is_usable(cuda):
    """tracker.py:146-149 with a motion model whose compute_log_likelihoods is None (tangent kinds): when the only
    observer is skipped (cloud beyond the frame) no likelihood exists at all and the weights of the last resampling
    stay in place — they are not reset to uniform."""
    import scenes

    scene = synthetic.nadir_scene(seed=6, n_points=2, n_particles=256, n_frames=6, imgsz=(320, 240), margin_px=100,
                                  velocity_sigma=0.3, kind="tangent_cartesian")
    scenes.add_gridded_dem(scene)
    scene.points[0, 0] = (320 / 2 - 24) * 0.2  # template fits, the growing cloud does not
    scene.motion["vxy"] = (2.0, 0.0)            # 10 px / day towards the edge
    tracks, ref, _ = run_both(scene, 21, "stream", return_particles=True)
    assert tracks.errors[0] is None and tracks.warnings[0] is not None
    skipped = (ref.skipped[0] == 2).any(axis=1)
    assert skipped.sum() == len(tracks.warnings[0]) > 0
    # at a skipped time the reported weights are a resampling of the previous ones: not all equal
    t_skip = int(np.nonzero(skipped)[0][0])
    assert np.ptp(ref.weights[0, t_skip]) > 0 and np.ptp(tracks.weights[0, t_skip]) > 0
    np.testing.assert_allclose(tracks.weights[0, t_skip], ref.weights[0, t_skip], rtol=1e-4)
    assert_close_to_oracle(tracks, ref)


@pytest.mark.parametrize("kind", ["cartesian", "cylindrical", "tangent_cartesian", "tangent_cylindrical"])
def test_stand_alone_evolve_particles_matches_the_oracle(cuda, kind):
    """``Motion.evolve_particles`` (gb_evolve) for every built-in model against the oracle's restatement of
    motion.py:165-179, 285-311, 392-420, 507-522 on the same draws; tangent models on a gridded DEM."""
    import glimpse_b200 as gb
    import scenes

    scene = synthetic.nadir_scene(seed=31, n_points=1, n_particles=500, n_frames=2, imgsz=(320, 240), margin_px=100, kind=kind)
    if kind.startswith("tangent"):
        scenes.add_gridded_dem(scene)
    _, models = synthetic.build(scene, gb)
    _, specs, _, _ = helpers.oracle_inputs(scene)
    np.random.seed(3)
    ps = orc.init_particles(specs[0])
    mine, ref = ps.copy(), ps.copy()
    dt = datetime.timedelta(days=1.5)
    np.random.seed(4)
    models[0].evolve_particles(mine, dt)
    np.random.seed(4)
    orc.evolve_particles(specs[0], ref, 1.5)
    np.testing.assert_allclose(mine, ref, rtol=1e-13, atol=1e-13)
    if kind.startswith("tangent"):
        far = ps.copy()
        far[:, 0] += 1e4  # off the DEM: Raster.sample raises (raster.py:961-973)
        with pytest.raises(ValueError, match="out of bounds"):
            models[0].evolve_particles(far, dt)


def test_kernel_timing_reports_every_kernel_of_the_streaming_flow(cuda):
    """gb_kernel_timing / gb_kernel_timing_read (include/glimpse_b200.h): CUDA-event durations per kernel kind."""
    import ctypes as C

    import glimpse_b200 as gb
    from glimpse_b200 import _lib

    scene = synthetic.nadir_scene(seed=2, n_points=8, n_particles=1000, n_frames=6, imgsz=(320, 240), margin_px=90)
    observers, models = synthetic.build(scene, gb)
    lib = _lib.load()
    _lib.check(lib.gb_kernel_timing(1))
    try:
        tracks = gb.Tracker(observers, seed=3).track(models, tile_size=scene.tile_size)
        ms, n = (C.c_double * 8)(), (C.c_int64 * 8)()
        _lib.check(lib.gb_kernel_timing_read(ms, n, 8))
    finally:
        _lib.check(lib.gb_kernel_timing(0))
    assert all(e is None for e in tracks.errors)
    # activity, surface, weights, resample+propagate, finalize, init, template, publish
    # per batch of points: one launch per time for the first three, one per update (5 of the 6 times) for the others
    assert list(n)[5:7] == [1, 1] and n[3] == n[4] and n[3] % 6 == 0 and n[1] == n[2] == n[7] == n[3] // 6 * 5 and 0 < n[0] <= n[3]
    assert all(ms[k] > 0 for k in range(8))
    _lib.check(lib.gb_kernel_timing_read(ms, n, 8))
    assert sum(n) == 0  # switching the timer off clears it


@pytest.mark.parametrize("rng", ["philox", "numpy"])
def test_blocks_of_points_give_the_same_track(cuda, rng):
    """A track that does not fit the device runs as consecutive blocks of points (Tracker.max_points forces it here):
    same results bit for bit, with the device draws (keyed by the global point index) and with the reference's draw
    sequence (consumed block after block in the reference's order)."""
    import glimpse_b200 as gb

    scene = synthetic.nadir_scene(seed=31, n_points=11, n_particles=500, n_frames=6, imgsz=(400, 300), margin_px=100)
    observers, models = synthetic.build(scene, gb)
    runs = []
    for max_points in (None, 4, 1):
        np.random.seed(77)
        tracker = gb.Tracker(observers, seed=5, rng=rng, max_points=max_points)
        tracks = tracker.track(models, tile_size=scene.tile_size, return_particles=(max_points != 1))
        assert all(e is None for e in tracks.errors)
        assert tracker.last_run.get("sessions", 1) == {None: 1, 4: 3, 1: 11}[max_points]
        runs.append((tracks, tracker))
    for tracks, tracker in runs[1:]:
        np.testing.assert_array_equal(tracks.means, runs[0][0].means)
        np.testing.assert_array_equal(tracks.sigmas, runs[0][0].sigmas)
        np.testing.assert_array_equal(tracker.particles, runs[0][1].particles)  # state of the last point, as the reference leaves it
    np.testing.assert_array_equal(runs[1][0].particles, runs[0][0].particles)
    assert len(runs[1][1].last_run["window_width"]) == len(runs[0][1].last_run["window_width"])


@pytest.mark.parametrize("method", ["systematic", "choice", "residual"])
@pytest.mark.parametrize("slots,batch", [(1, 7), (4, 2), (4, 1), (2, 5)])
def test_the_batch_plan_does_not_change_the_track(cuda, monkeypatch, slots, batch, method):
    """gb_track cuts the points into batches that advance on their own streams (one batch for few points, up to four): points are
    independent and Philox counters are global, so every plan gives bit-identical results — also with an observer that starts
    later (templates join the batches) and a point that fails on the way.  'systematic' runs the pipelined flow, 'choice' and
    'residual' the step-by-step one."""
    import glimpse_b200 as gb

    scene = synthetic.nadir_scene(seed=31, n_points=7, n_particles=700, n_frames=7, imgsz=(400, 300), margin_px=100)
    scenes.add_second_observer(scene)
    scene.points[3] = (1.0e4, 1.0e4)  # far outside every frame: fails at its template
    observers, models = synthetic.build(scene, gb)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        base = gb.Tracker(observers, seed=9, resample_method=method).track(models, tile_size=scene.tile_size, return_covariances=True,
                                                                         return_particles=True)
        monkeypatch.setenv("GB_STREAM_SLOTS", str(slots))
        monkeypatch.setenv("GB_STREAM_BATCH", str(batch))
        tracker = gb.Tracker(observers, seed=9, resample_method=method)
        other = tracker.track(models, tile_size=scene.tile_size, return_covariances=True, return_particles=True)
    plan = tracker.last_run["plan"]
    assert plan["stream_slots"] == slots and plan["stream_batch"] == batch
    assert base.errors[3] is not None and sum(e is not None for e in base.errors) == 1
    assert [type(e) for e in other.errors] == [type(e) for e in base.errors]
    np.testing.assert_array_equal(other.means, base.means)
    np.testing.assert_array_equal(other.covariances, base.covariances)
    np.testing.assert_array_equal(other.particles, base.particles)


def test_kernel_launches_of_the_step_by_step_flow(cuda, monkeypatch):
    """Tracker.last_run['kernel_launches'] of a 'choice' track counts what gb_track launched: per batch of points and update
    k_s0 k_s1 k_s2 k_s3 k_s4c_scan k_s4c_gather k_s5, and k_init and k_template at the first time."""
    import glimpse_b200 as gb

    scene = synthetic.nadir_scene(seed=2, n_points=3, n_particles=500, n_frames=4, imgsz=(320, 240), margin_px=90)
    observers, models = synthetic.build(scene, gb)
    monkeypatch.setenv("GB_STREAM_SLOTS", "2")
    monkeypatch.setenv("GB_STREAM_BATCH", "2")
    tracker = gb.Tracker(observers, seed=3, resample_method="choice")
    tracks = tracker.track(models, tile_size=scene.tile_size)
    assert all(e is None for e in tracks.errors)
    batches, updates = 2, 3
    assert tracker.last_run["kernel_launches"] == 7 * batches * updates + 1 + 1


@pytest.mark.parametrize("kind", ["cartesian", "cylindrical", "tangent_cartesian", "tangent_cylindrical"])
def test_stand_alone_initialize_and_log_likelihoods_match_the_oracle(cuda, kind):
    """The rest of the Motion protocol (motion.py:13-89) as stand-alone calls: ``initialize_particles``
    (gb_init_particles) and ``compute_log_likelihoods`` (gb_motion_log_likelihoods) against the oracle's restatements of
    motion.py:149-163, 260-283, 378-390, 485-505 and 181-204 on the same draws, on a gridded DEM with a gridded sigma."""
    import glimpse_b200 as gb
    import scenes

    scene = synthetic.nadir_scene(seed=33, n_points=1, n_particles=700, n_frames=2, imgsz=(320, 240), margin_px=100, kind=kind)
    scenes.add_gridded_dem(scene)
    _, models = synthetic.build(scene, gb)
    _, specs, _, _ = helpers.oracle_inputs(scene)
    np.random.seed(5)
    mine = models[0].initialize_particles()
    np.random.seed(5)
    ref = orc.init_particles(specs[0])
    assert mine.shape == ref.shape == (700, 6)
    np.testing.assert_allclose(mine, ref, rtol=1e-13, atol=1e-13)
    ll, ll_ref = models[0].compute_log_likelihoods(ref), orc.surface_log_likelihood(specs[0], ref)
    if kind.startswith("tangent"):
        assert ll is None and ll_ref is None
    else:
        assert ll.shape == (700,) and (ll_ref > 0).any()
        np.testing.assert_allclose(ll, ll_ref, rtol=1e-12, atol=1e-300)
    far = ref.copy()
    far[:, 0] += 1e4  # off the DEM: Raster.sample raises (raster.py:961-973)
    if not kind.startswith("tangent"):
        with pytest.raises(ValueError, match="out of bounds"):
            models[0].compute_log_likelihoods(far)
    models[0].xy = (1e4, 0.0)
    with pytest.raises(ValueError, match="out of bounds"):
        models[0].initialize_particles()


def _dispersing_scene(n_points, n_particles):
    """A weakly informative observer (sigma = 5) and a wide velocity prior (2 m/d = 10 px/d): the particle cloud, and with it
    the search window, grows by ~60 px per frame — far beyond the default capacity of template + 191 px."""
    scene = synthetic.nadir_scene(seed=41, n_points=n_points, n_particles=n_particles, n_frames=9, imgsz=(1400, 1000), margin_px=560)
    scene.observers[0].sigma = 5.0
    scene.motion.update(vxyz_sigma=(2.0, 2.0, 0.0))
    return scene


def test_search_windows_of_several_hundred_pixels_match_the_oracle(cuda):
    """Windows up to ~500 px (SSE surfaces beyond 256 cells per axis, worked on in global memory) with the reference's draws
    against the oracle, which calls OpenCV / FITPACK on the same windows."""
    import glimpse_b200 as gb

    scene = _dispersing_scene(1, 400)
    observers, models = synthetic.build(scene, gb)
    tracker = gb.Tracker(observers, rng="numpy", window_margin=1000)
    np.random.seed(12)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        tracks = tracker.track(models, tile_size=scene.tile_size, return_particles=True)
    assert tracks.errors[0] is None, tracks.errors
    assert tracker.last_run["window_width"].max() > 300
    obs, specs, taus, index = helpers.oracle_inputs(scene)
    np.random.seed(12)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref = orc.track(obs, specs, taus, index, tile_size=scene.tile_size, return_particles=True, raise_errors=True)
    same = np.isclose(tracks.particles, ref.particles, rtol=0, atol=1e-9).all(axis=3)
    assert 1.0 - same.mean() < 0.02
    assert np.nanmax(np.abs(tracks.means - ref.means) / np.maximum(ref.sigmas, 1e-12)) < 0.05


def test_points_that_outgrow_the_window_capacity_are_run_again(cuda):
    """Default capacity (template + 191 px): the dispersing points stop with GB_ST_WINDOW_TOO_LARGE and are tracked again with
    the largest capacity; the counter-based draws make the result identical to a run planned with that capacity from the
    start.  With the reference's draw sequence (not replayable) the error is reported."""
    import glimpse_b200 as gb

    scene = _dispersing_scene(3, 400)
    observers, models = synthetic.build(scene, gb)
    wide = gb.Tracker(observers, seed=3, window_margin=1000).track(models, tile_size=scene.tile_size)
    assert all(e is None for e in wide.errors)
    tracker = gb.Tracker(observers, seed=3)
    tracks = tracker.track(models, tile_size=scene.tile_size)
    assert all(e is None for e in tracks.errors), tracks.errors
    assert tracker._rerun_points == [0, 1, 2]
    np.testing.assert_array_equal(tracks.means, wide.means)
    np.testing.assert_array_equal(tracks.sigmas, wide.sigmas)
    blocked = gb.Tracker(observers, seed=3, max_points=2).track(models, tile_size=scene.tile_size)
    np.testing.assert_array_equal(blocked.means, wide.means)
    np.random.seed(1)
    kept = gb.Tracker(observers, rng="numpy").track(models, tile_size=scene.tile_size)
    assert all(isinstance(e, MemoryError) for e in kept.errors)
    assert np.isfinite(kept.means[:, 1]).all() and np.isnan(kept.means[:, -1]).all()


def test_models_with_their_own_particle_counts(cuda):
    """tracker.py:328: every motion model carries its own n.  Points are tracked group by group (one device session per
    particle count) and come back in their order; a group's results equal those of tracking that group alone."""
    import glimpse_b200 as gb

    scene = synthetic.nadir_scene(seed=6, n_points=6, n_particles=500, n_frames=5, imgsz=(320, 240), margin_px=100)
    observers, models = synthetic.build(scene, gb)
    for i in (1, 4):
        models[i].n = 800
    tracker = gb.Tracker(observers, seed=21)
    tracks = tracker.track(models, tile_size=scene.tile_size, return_particles=True)
    assert all(e is None for e in tracks.errors) and tracks.means.shape == (6, 5, 6)
    assert [p.shape for p in tracks.particles] == [(5, 800 if i in (1, 4) else 500, 6) for i in range(6)]
    assert np.isfinite(tracks.means).all() and np.all(np.abs(tracks.vxyz[:, -1, 0] - scene.truth_velocity[0]) < 0.15)
    first = gb.Tracker(observers, seed=21).track([models[i] for i in (0, 2, 3, 5)], tile_size=scene.tile_size)
    np.testing.assert_array_equal(tracks.means[[0, 2, 3, 5]], first.means)
    second = gb.Tracker(observers, seed=22).track([models[i] for i in (1, 4)], tile_size=scene.tile_size)
    np.testing.assert_array_equal(tracks.means[[1, 4]], second.means)
    assert tracker.seed == 21
