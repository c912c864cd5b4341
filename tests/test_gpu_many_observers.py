"""Calls with more than eight observers, up to eight of them with a frame at the same time.

The kernels take a time step's cameras from a slot table: one slot per observer with a frame at that time, in ascending
observer order.  Checked here: free-running tracks against the oracle, every update teacher-forced through
``gb_track_step`` (including a time whose slots hold observers 2, 7 and 10), bit-identity with the one-slot-per-observer
path of a call of eight observers, and sharding over two GPUs."""
import datetime
import os
import socket
import subprocess
import sys
import textwrap
import warnings

import numpy as np
import pytest

import helpers
from glimpse_b200 import synthetic
from oracle import tracker_oracle as orc
from test_gpu_edge import assert_close_to_oracle
from test_gpu_track import (MOMENT_REL, SAMPLED_ABS, SEARCH_TOL, SSE_REL_CV2, SSE_REL_EXACT, UV_TOL_PX, WEIGHT_REL,
                            make_session)

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# observers with a frame at each time: at most three of twelve, the sets change every one or two frames, templates start at
# 0, 2, 4, 5, 6 and 7, times 2-3 have slots (2, 7, 10), which k_s4p's generic loop serves from its third slot on, and time 8
# has one slot more than time 7 (k_s4p must project into the slots of the next time, not of its own)
TWELVE = [{0, 1, 4}, {0, 1, 4}, {2, 7, 10}, {2, 7, 10}, {3, 5, 11}, {3, 6, 11}, {5, 6, 8}, {8, 9}, {1, 4, 9}]
# eleven observers, eight of them at time 1
ELEVEN = [{0, 1}, {0, 1, 2, 3, 4, 5, 6, 7}, {3, 8, 9, 10}, {1, 2, 8, 9}, {4, 5, 6, 10}, {0, 7, 10}]


def station(base, times, style, sigma):
    """One observer showing the base frames of ``times``: 'grey' as they are, 'rolled' turned 180 deg into RGB (as
    ``scenes.add_second_observer``), 'u16' as uint16 with sub-grey-level detail (the ranked tile path)."""
    frames, cams = [], []
    rng = np.random.RandomState(5)
    for t in times:
        g, vec = base.frames[t], base.cams[t].copy()
        if style == "rolled":
            g = g[::-1, ::-1]
            g = np.stack([g, np.roll(g, 1, axis=1), np.roll(g, 1, axis=0)], axis=2)
            vec[3:6] = (0.0, -90.0, 180.0)
            vec[18:20] = 0.0
        elif style == "u16":
            g = g.astype(np.uint16) * 200 + rng.randint(0, 200, g.shape).astype(np.uint16)
        frames.append(np.ascontiguousarray(g))
        cams.append(vec)
    return synthetic.ObserverScene(frames, np.array(cams), [base.datetimes[t] for t in times], sigma=sigma)


def schedule_scene(schedule, n_obs, styles=None, n_points=3, n_particles=256, seed=31, **scene_kw):
    """A scene whose observer o has the base scene's frame t exactly when o is in ``schedule[t]``."""
    kw = dict(imgsz=(320, 240), margin_px=100)
    kw.update(scene_kw)
    scene = synthetic.nadir_scene(seed=seed, n_points=n_points, n_particles=n_particles, n_frames=len(schedule), **kw)
    base = scene.observers[0]
    styles = styles or {}
    scene.observers = [station(base, [t for t, s in enumerate(schedule) if o in s], styles.get(o, "rolled" if o % 3 == 1 else "grey"),
                               0.3 + 0.02 * o) for o in range(n_obs)]
    return scene


def mask_for(n_points, n_obs, hidden):
    mask = np.ones((n_points, n_obs), dtype=bool)
    for p, obs in hidden.items():
        mask[p, list(obs)] = False
    return mask


CASES = {
    "twelve": dict(scene=lambda: schedule_scene(TWELVE, 12)),
    "eleven_eight_at_once": dict(scene=lambda: schedule_scene(ELEVEN, 11, seed=33)),
    "observer_mask": dict(scene=lambda: schedule_scene(TWELVE, 12, seed=35), observer_mask=mask_for(3, 12, {0: {2, 7}, 1: {0, 1}, 2: {3, 10}})),
    "covariances_particles": dict(scene=lambda: schedule_scene(TWELVE, 12, seed=37), return_covariances=True, return_particles=True),
    "uint16_observer": dict(scene=lambda: schedule_scene(TWELVE, 12, styles={7: "u16"}, seed=39)),
    "template_33x32": dict(scene=lambda: schedule_scene(TWELVE, 12, n_points=2, seed=41, imgsz=(400, 300), margin_px=110,
                                                        tile_size=(33, 32))),
    "choice": dict(scene=lambda: schedule_scene(TWELVE, 12, seed=43), resample_method="choice"),
}


def slots_of(scene):
    _, _, _, index = helpers.oracle_inputs(scene)
    return int((index >= 0).sum(axis=1).max())


@pytest.mark.parametrize("name", list(CASES))
def test_many_observers_match_oracle(cuda, name):
    import glimpse_b200 as gb

    case = CASES[name]
    scene = case["scene"]()
    kw = {k: case[k] for k in ("observer_mask", "return_covariances", "return_particles") if k in case}
    method = case.get("resample_method", "systematic")
    observers, models = synthetic.build(scene, gb)
    tracker = gb.Tracker(observers, rng="numpy", resample_method=method)
    np.random.seed(19)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        tracks = tracker.track(models, tile_size=scene.tile_size, **kw)
    obs, specs, taus, index = helpers.oracle_inputs(scene)
    np.random.seed(19)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref = orc.track(obs, specs, taus, index, tile_size=scene.tile_size, resample_method=method, **kw)
    assert len(observers) > 8
    assert tracker.last_run["plan"]["n_observers"] == slots_of(scene)
    assert all(e is None for e in tracks.errors), tracks.errors
    assert all(e is None for e in ref.errors), ref.errors
    assert_close_to_oracle(tracks, ref, sig_tol=1e-3)
    if kw.get("return_covariances"):
        scale = np.sqrt(np.einsum("ptii->pti", ref.sigmas))
        ok = ~np.isnan(scale[..., 0])
        d = np.abs(tracks.covariances - ref.sigmas)[ok] / np.maximum(scale[ok][:, :, None] * scale[ok][:, None, :], 1e-12)
        assert float(d.max()) < 1e-3
    if kw.get("return_particles"):
        assert tracks.particles.shape == ref.particles.shape
        same = np.isclose(tracks.particles, ref.particles, rtol=0, atol=1e-6).all(axis=3)
        assert same.mean() > 0.99, same.mean()
    # Tracker.templates (the last point's) stays indexed by observer: one per observer that saw the point
    mask = kw.get("observer_mask", np.ones((len(models), len(observers)), dtype=bool))
    assert [t is not None for t in tracker.templates] == list(mask[-1])


def test_many_observers_refuse_nine_at_once(cuda):
    import glimpse_b200 as gb

    schedule = [{0, 1, 5, 6}, {0, 1, 2, 7, 8}, set(range(1, 10)), {3, 4, 9}]
    scene = schedule_scene(schedule, 10)
    observers, models = synthetic.build(scene, gb)
    with pytest.raises(NotImplementedError, match="time index 2"):
        gb.Tracker(observers, rng="numpy").track(models, tile_size=scene.tile_size)


def oracle_golden(scene, seed):
    """The oracle's intermediates in the key layout of the ``track_*`` fixtures (as ``test_gpu_large_template``)."""
    obs, models, taus, idx = helpers.oracle_inputs(scene)
    np.random.seed(seed)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        res = orc.track(obs, models, taus, idx, tile_size=scene.tile_size, return_particles=True, trace=True)
    steps = [s for s in res.trace if "indices" in s]
    g = {"images": idx, "seed": seed, "n_steps": len(steps), "means": res.means, "sigmas": res.sigmas}
    for i, s in enumerate(steps):
        for key in ("evolved", "weights", "u", "indices"):
            g[f"step{i}.{key}"] = np.asarray(s[key])
        for o, rec in s.get("obs", {}).items():
            for key, val in rec.items():
                g[f"step{i}.obs.{o}.{key}"] = np.asarray(val)
    templates = {}
    for t in res.templates:
        templates.setdefault(int(t["p"]), {})[int(t["obs"])] = np.asarray(t["tile"])
    return g, templates


def test_many_observers_step_teacher_forced(cuda):
    """Every update of the twelve-observer scene forced through gb_track_step: the dumps stay [P][O] by observer, while the
    kernels work on the slots of each time (at t = 2, 3 the slots hold observers 2, 7 and 10)."""
    from glimpse_b200 import _lib

    torch = cuda
    scene = schedule_scene(TWELVE, 12, n_points=2, seed=45)
    g, templates = oracle_golden(scene, 4545)
    session, _ = make_session(scene, {}, g)
    assert session.O == 12 and session.plan.n_observers == 3
    P, N, O = session.P, session.N, session.O
    per = int(g["n_steps"]) // P
    dev = session.device
    session.run()
    torch.cuda.synchronize()
    assert (session.buf["status"].cpu().numpy() == 0).all()
    cap = 200 * 200
    worst = dict(uv=0.0, search=0.0, sse_cv2=0.0, sse_exact=0.0, sampled=0.0, weights=0.0, mean=0.0, sigma=0.0)
    slot_sets = set()

    def upd(key, values):
        v = float(np.max(values))
        assert np.isfinite(v), f"{key}: non-finite difference (missing or NaN output)"
        worst[key] = max(worst[key], v)

    for s in range(per):
        t = int(session.first[0]) + 1 + s
        evolved = np.stack([g[f"step{p * per + s}.evolved"] for p in range(P)])
        weights_ref = np.stack([g[f"step{p * per + s}.weights"] for p in range(P)])
        u_ref = np.array([float(np.atleast_1d(g[f"step{p * per + s}.u"])[0]) for p in range(P)])
        session.buf["uniforms"][:, t - 1 - int(session.first[0])] = torch.as_tensor(u_ref).to(dev)
        f_ev = torch.as_tensor(np.ascontiguousarray(evolved.transpose(0, 2, 1))).to(dev)
        dump = {
            "uv": torch.full((P, O, N, 2), float("nan"), dtype=torch.float64, device=dev),
            "box": torch.full((P, O, 4), -1, dtype=torch.int32, device=dev),
            "search": torch.zeros((P, O, cap), dtype=torch.float32, device=dev),
            "sse": torch.zeros((P, O, cap), dtype=torch.float32, device=dev),
            "sampled": torch.zeros((P, O, N), dtype=torch.float64, device=dev),
            "weights": torch.zeros((P, N), dtype=torch.float64, device=dev),
            "indices": torch.full((P, N), -1, dtype=torch.int32, device=dev),
        }
        io = _lib.gb_stage_io()
        io.force_evolved = f_ev.data_ptr()
        io.dump_uv, io.dump_box = dump["uv"].data_ptr(), dump["box"].data_ptr()
        io.dump_search, io.dump_sse = dump["search"].data_ptr(), dump["sse"].data_ptr()
        io.dump_sampled, io.dump_weights = dump["sampled"].data_ptr(), dump["weights"].data_ptr()
        io.dump_indices = dump["indices"].data_ptr()
        io.dump_cap = cap
        session.buf["status"].zero_()
        session.step(t, io)
        torch.cuda.synchronize()
        assert (session.buf["status"].cpu().numpy() == 0).all()
        got = {k: v.cpu().numpy() for k, v in dump.items()}
        slot_sets.add(tuple(sorted(TWELVE[t])))
        for p in range(P):
            rec = f"step{p * per + s}."
            used = [o for o in range(O) if f"{rec}obs.{o}.uv" in g]
            assert set(used) <= TWELVE[t] and used
            for o in range(O):
                key = f"{rec}obs.{o}."
                if o not in used:
                    assert (got["box"][p, o] == -1).all() and np.isnan(got["uv"][p, o]).all()  # no slot wrote this observer's rows
                    continue
                upd("uv", np.abs(got["uv"][p, o] - g[key + "uv"]))
                np.testing.assert_array_equal(got["box"][p, o], g[key + "box"])
                search_ref = g[key + "search"]
                sv, su = search_ref.shape
                upd("search", np.abs(got["search"][p, o, : sv * su].reshape(sv, su) - search_ref.astype(np.float32)))
                sse_ref = g[key + "sse"]
                mv, mu = sse_ref.shape
                sse = got["sse"][p, o, : mv * mu].reshape(mv, mu)
                upd("sse_cv2", np.abs(sse - sse_ref) / np.maximum(sse_ref, 1e-3))
                exact = orc.ssd_surface(search_ref, templates[p][o], exact=True)
                upd("sse_exact", np.abs(sse - exact) / np.maximum(exact, 1e-3))
                upd("sampled", np.abs(got["sampled"][p, o] - g[key + "sampled"]))
            upd("weights", np.abs(got["weights"][p] - weights_ref[p]) / weights_ref[p])
        f_w = torch.as_tensor(weights_ref).to(dev)
        io2 = _lib.gb_stage_io()
        io2.force_evolved, io2.force_weights = f_ev.data_ptr(), f_w.data_ptr()
        io2.dump_indices = dump["indices"].data_ptr()
        session.step(t, io2)
        torch.cuda.synchronize()
        idx = dump["indices"].cpu().numpy()
        means = session.buf["means"].cpu().numpy()
        sig = session.buf["sig"].cpu().numpy()
        for p in range(P):
            np.testing.assert_array_equal(idx[p], g[f"step{p * per + s}.indices"])
            m_ref = g["means"][p, t]
            upd("mean", np.abs(means[p, t] - m_ref) / np.maximum(np.abs(m_ref), 1e-3))
            s_ref = g["sigmas"][p, t]
            ok = s_ref > 0
            upd("sigma", np.abs(sig[p, t][ok] - s_ref[ok]) / s_ref[ok])
    print("worst", {k: float(v) for k, v in worst.items()})
    assert (2, 7, 10) in slot_sets
    assert worst["uv"] <= UV_TOL_PX
    assert worst["search"] <= SEARCH_TOL
    assert worst["sse_cv2"] <= SSE_REL_CV2
    assert worst["sse_exact"] <= SSE_REL_EXACT
    assert worst["sampled"] <= SAMPLED_ABS
    assert worst["weights"] <= WEIGHT_REL
    assert worst["mean"] <= MOMENT_REL
    assert worst["sigma"] <= 1e-7


EIGHT = [{0, 1, 4}, {0, 1, 4}, {2, 5, 7}, {2, 5, 7, 3}, {3, 5, 6}, {3, 6}, {1, 5, 6}, {0, 6, 7}]
EXTRA_AT = (0, 5, 9, 11)  # positions of the added observers in the twelve-observer call


def with_unmatched_observers(scene):
    """The scene's observers with four more inserted at EXTRA_AT, whose frames are 12 h off every time of the track."""
    out = list(scene.observers)
    for k, at in enumerate(EXTRA_AT):
        src = scene.observers[k % len(scene.observers)]
        off = [d + datetime.timedelta(hours=12) for d in src.datetimes]
        out.insert(at, synthetic.ObserverScene([f.copy() for f in src.frames], src.cams.copy(), off, sigma=0.5))
    return out


def philox_session(scene, observers_scene, seed, return_particles=True):
    import glimpse_b200 as gb
    from glimpse_b200.session import Session

    scene_o = synthetic.Scene(observers_scene, scene.points, scene.motion, scene.n_particles, scene.tile_size, scene.time_unit)
    observers, models = synthetic.build(scene_o, gb)
    tracker = gb.Tracker(observers, seed=seed)
    datetimes = scene.datetimes
    matching = tracker.match_datetimes(datetimes)
    index = np.array([[-1 if v is None else int(v) for v in row] for row in matching], dtype=np.int32)
    unit = scene.time_unit.total_seconds()
    taus = np.array([dt.total_seconds() / unit for dt in np.diff(datetimes)])
    mask = np.ones((len(models), len(observers)), dtype=bool)
    session = Session(tracker, models, index, taus, scene.tile_size, mask, return_particles=return_particles, seed=seed)
    session.run()
    out = session.fetch()
    return out, session, tracker, models


def test_slot_path_is_bit_identical_to_the_identity_path(cuda):
    """Eight observers (one slot each) against the same eight plus four whose frames match no time of the track (slots of
    the observers with a frame): rng='philox' with one seed gives the same bits, and the added observers are flagged
    GB_OBS_NO_IMAGE wherever a point is updated."""
    import glimpse_b200 as gb
    from glimpse_b200 import _lib

    scene = schedule_scene(EIGHT, 8, n_points=3, n_particles=700, seed=47)
    a, sa, _, _ = philox_session(scene, scene.observers, 4747)
    b, sb, _, _ = philox_session(scene, with_unmatched_observers(scene), 4747)
    assert sa.plan.n_observers == 8 and sb.O == 12 and sb.plan.n_observers == 4
    assert (a["status"] == 0).all()
    for key in ("means", "sigmas", "particles", "weights", "status", "status_time"):
        np.testing.assert_array_equal(a[key], b[key], err_msg=key)
    keep = [o for o in range(12) if o not in EXTRA_AT]
    np.testing.assert_array_equal(a["obs_flags"], b["obs_flags"][:, :, keep])
    updated = np.zeros(a["obs_flags"].shape[:2], dtype=bool)
    for p in range(sa.P):
        updated[p, sa.first[p] + 1: sa.last[p] + 1] = True
    extra = b["obs_flags"][:, :, list(EXTRA_AT)]
    assert (extra[updated] == _lib.GB_OBS_NO_IMAGE).all()
    assert (extra[~updated] == 0).all()
    # the public entry point with explicit datetimes: same means
    observers8, models = synthetic.build(scene, gb)
    scene12 = synthetic.Scene(with_unmatched_observers(scene), scene.points, scene.motion, scene.n_particles, scene.tile_size,
                              scene.time_unit)
    observers12, _ = synthetic.build(scene12, gb)
    t8 = gb.Tracker(observers8, seed=4747).track(models, datetimes=scene.datetimes, tile_size=scene.tile_size)
    t12 = gb.Tracker(observers12, seed=4747).track(models, datetimes=scene.datetimes, tile_size=scene.tile_size)
    np.testing.assert_array_equal(t8.means, t12.means)
    np.testing.assert_array_equal(t8.sigmas, t12.sigmas)
    np.testing.assert_array_equal(t8.tracker.particles, t12.tracker.particles)


def test_weights_sum_the_observers_in_observer_order(cuda):
    """k_s3_weights sums the observers' log-likelihoods in slot order; the slots list the observers of a time in ascending
    order, the order of the one-slot-per-observer path (and of the reference).  A sum in another order differs in the last
    bits of the log-likelihood, which reach a weight only now and then: exp(-ll) takes its fraction through float32.  So
    the weights of many particles with large log-likelihoods (small pixel sigmas) are compared: 200 points x 100 000
    particles forced into every update of both calls through gb_track_step, weights dumped, bit for bit."""
    from glimpse_b200 import _lib

    torch = cuda
    scene = schedule_scene(EIGHT, 8, n_points=200, n_particles=100000, seed=51)
    for o, obs in enumerate(scene.observers):
        obs.sigma = 0.08 + 0.01 * o
    a, sa, _, _ = philox_session(scene, scene.observers, 5151, return_particles=False)
    b, sb, _, _ = philox_session(scene, with_unmatched_observers(scene), 5151, return_particles=False)
    assert sa.plan.n_observers == 8 and sb.plan.n_observers == 4
    np.testing.assert_array_equal(a["means"], b["means"])
    P, N = sa.P, sa.N
    final = sa.buf["state_b"] if int(sa.last[0]) & 1 else sa.buf["state_a"]
    forced = final.clone()  # (P, 6, N): the last particles of the track, forced into every update
    for t in range(1, sa.T):
        got = []
        for session in (sa, sb):
            w = torch.zeros((P, N), dtype=torch.float64, device=session.device)
            io = _lib.gb_stage_io()
            io.force_evolved, io.dump_weights = forced.data_ptr(), w.data_ptr()
            session.buf["status"].zero_()
            session.step(t, io)
            torch.cuda.synchronize()
            got.append(w)
        assert torch.equal(got[0], got[1]), (t, int((got[0] != got[1]).sum()))


WORKER = textwrap.dedent('''
    import os, sys
    import numpy as np
    import torch
    import torch.distributed as dist
    sys.path.insert(0, sys.argv[1]); sys.path.insert(0, os.path.join(sys.argv[1], "tests"))
    import glimpse_b200 as gb
    from glimpse_b200 import synthetic
    from test_gpu_many_observers import TWELVE, schedule_scene
    rank = int(os.environ["RANK"]); torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ["LOCAL_RANK"])))
    scene = schedule_scene(TWELVE, 12, n_points=5, n_particles=1000, seed=49)
    observers, models = synthetic.build(scene, gb)
    sharded = gb.Tracker(observers, seed=13).track(models, tile_size=scene.tile_size, return_particles=True)
    alone = gb.Tracker(observers, seed=13, distributed=False).track(models, tile_size=scene.tile_size, return_particles=True)
    assert all(e is None for e in alone.errors)
    np.testing.assert_array_equal(sharded.means, alone.means)
    np.testing.assert_array_equal(sharded.sigmas, alone.sigmas)
    np.testing.assert_array_equal(sharded.particles, alone.particles)
    dist.barrier(); dist.destroy_process_group()
    print("rank", rank, "ok")
''')


def test_many_observers_two_ranks_match_one_gpu(cuda, tmp_path):
    if cuda.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), str(script), ROOT]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-4000:]
    assert out.stdout.count("ok") == 2
