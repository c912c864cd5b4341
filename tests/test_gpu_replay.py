"""Every update of production ``Tracker.track`` runs (the pipelined flow: k_s2_surface -> k_s3_weights -> k_s3b_publish ->
k_s4p_resample_propagate -> k_s5p_finalize) replayed in float64 from the track's own outputs (tests/replay.py), at 2 to
1 000 001 particles: 1 to 1 303 blocks per point, odd N, stratified resampling, carried, uniform, DEM-only and observed
updates, a late-starting point, a failed point in a batch of active points, a call mixing cartesian, cylindrical and
tangent points over three observers with its datetimes backwards, batches of points running concurrently on up to four side
streams.  The same for the step-by-step flow (k_s1_propagate -> k_s2_surface -> k_s3_weights -> k_s4c_scan or
k_s4r_residual -> k_s4c_gather -> k_s5_finalize) that runs the choice and residual resamplers.  And the resampler at the
edge uniforms 0, 2^-30, 1/2 and 1 - 2^-53, supplied as draws."""
import numpy as np
import pytest

import helpers
import philox
import replay
from glimpse_b200 import synthetic

pytestmark = pytest.mark.gpu

SEED = replay.SEED


def record_sessions(monkeypatch):
    """Make ``Tracker.track``'s sessions keep what they fetched and their realised window sizes."""
    from glimpse_b200 import session as session_mod

    kept = []

    class Recording(session_mod.Session):
        def fetch(self, gather=None):
            out = super().fetch(gather)
            kept.append((out, self.buf["window"].cpu().numpy()))
            return out

    monkeypatch.setattr(session_mod, "Session", Recording)
    return kept


def check_final_state(tracker, res):
    P = res["particles"].shape[0]
    last = int(np.nonzero(~np.isnan(res["weights"][P - 1, :, 0]))[0][-1])
    assert np.array_equal(tracker.particles, res["particles"][P - 1, last])
    assert np.array_equal(tracker.weights, res["weights"][P - 1, last])


def track_and_replay(monkeypatch, name, method=None):
    """Tracker.track of a replay case (``method``: another resampler) and the replay of every update; returns (report,
    tracks)."""
    import glimpse_b200 as gb
    from glimpse_b200.session import point_span

    # one batch per point (two in the mixed call, so that its failing point shares a batch with an active one), four side
    # streams: the batches of a multi-point case run concurrently
    monkeypatch.setenv("GB_STREAM_BATCH", "2" if name == "mixed_three_obs" else "1")
    monkeypatch.setenv("GB_STREAM_SLOTS", "4")
    kept = record_sessions(monkeypatch)
    scene, mask, method, cov = replay.case(name, method=method)
    observers, models = replay.build(scene, gb)
    tracker = gb.Tracker(observers, seed=SEED, resample_method=method)
    tracks = tracker.track(models, datetimes=replay.datetimes(scene), tile_size=scene.tile_size, observer_mask=mask,
                           return_particles=True, return_covariances=cov)
    assert len(kept) == 1
    res, windows = kept[0]
    np.testing.assert_array_equal(tracks.means, res["means"])
    inputs = replay.inputs(scene)
    first, last = point_span(inputs[3].astype(np.int32), mask)
    P = len(models)
    draws = philox.device_draws(SEED, range(P), first, last, scene.n_particles, [m.tangent for m in inputs[1]], method)
    rep = replay.replay_track(res, draws, inputs, method, mask, scene.tile_size, cov=cov, windows=windows)
    print(replay.summary(f"{name} ({method})", rep))
    check_final_state(tracker, res)
    assert rep["windows"] > 0
    if name.startswith("small_") or name == "mixed_three_obs":
        assert rep["failed points"] == 1 and tracks.errors[1] is not None
    if name == "mixed_three_obs":
        assert all(rep[f"{k} updates"] > 0 for k in replay.KINDS)
    if name == "cart_dem_floor":
        assert rep["dem updates"] == 4
    return rep, tracks


@pytest.mark.parametrize("name", replay.CASES)
def test_every_update_replays(cuda, monkeypatch, name):
    rep, _ = track_and_replay(monkeypatch, name)
    if name == "tan_carried_collapse":
        assert rep["children of one parent (observed)"] > 3 * replay.CHUNK and rep["carried updates"] == 2


@pytest.mark.parametrize("name,method", replay.STEP_CASES)
def test_every_step_flow_update_replays(cuda, monkeypatch, name, method):
    """The step-by-step flow of gb_track (choice, residual) replayed: k_s1_propagate for every particle (the pipelined cases'
    draws), k_s4c_scan's cumulative weights across up to 1 303 blocks, k_s4r_residual at up to 10^5 particles (every child
    searched at small_99005's uniform updates), k_s4c_gather and k_s5_finalize combining the moment partials."""
    rep, _ = track_and_replay(monkeypatch, name, method)
    if name == "tan_carried_collapse":  # a parent with more than three blocks of children, drawn in any order
        assert rep["children of one parent (observed)"] > 3 * replay.CHUNK and rep["carried updates"] == 2
    if name == "small_99005":
        assert rep["residual K = 0 (uniform)"] == rep["uniform updates"] > 0


EDGE_U = [0.0, 1 - 2.0 ** -53, 2.0 ** -30, 0.5]


@pytest.mark.parametrize("method", ["systematic", "stratified"])
@pytest.mark.parametrize("N", [1024, 131072, 1000, 10000])
def test_edge_uniforms(cuda, method, N):
    """Uniform updates (weights exactly 1) with supplied uniforms at the edges, one value per point: with N a power of two
    every cumulative weight and position is exact and the ancestors must equal np.searchsorted's bit for bit (no near-tie);
    at N = 1 000 and 10 000 the reference's cumsum is inexact and near-ties within 1e-12 are counted."""
    import glimpse_b200 as gb
    from glimpse_b200.session import Session, point_span

    scene = synthetic.nadir_scene(seed=66, n_points=len(EDGE_U), n_particles=N, n_frames=3, imgsz=(320, 240), margin_px=100)
    replay.interleave(scene)
    P, O = len(scene.points), len(scene.observers)
    mask = np.ones((P, O), dtype=bool)
    mask[:, O - 1] = False
    observers, models = synthetic.build(scene, gb)
    tracker = gb.Tracker(observers, resample_method=method, rng="numpy")
    inputs = helpers.oracle_inputs(scene)
    image_index = inputs[3].astype(np.int32)
    first, last = point_span(image_index, mask)
    S = int((last - first).max())
    rng = np.random.RandomState(N)
    init, step = rng.randn(P, N, 6), rng.randn(P, S, N, 3)
    u = np.asarray(EDGE_U)
    unif = np.broadcast_to(u[:, None, None], (P, S, N)).copy() if method == "stratified" else np.broadcast_to(u[:, None], (P, S)).copy()
    session = Session(tracker, models, image_index, inputs[2], scene.tile_size, mask, return_particles=True,
                      draws=(init, step, unif))
    session.run()
    res = session.fetch()
    assert (res["status"] == 0).all()
    rep = replay.replay_track(res, (init, step, unif), inputs, method, mask, scene.tile_size, windows=session.buf["window"].cpu().numpy())
    print(replay.summary(f"edge uniforms {method} N {N}", rep))
    assert rep["uniform updates"] == 2 * P
    if N & (N - 1) == 0:
        assert rep["near-ties (uniform)"] == 0
