"""The default ``rng='philox'`` path against the host restatement of its generator and against the reference.

The generator: the words, normals and uniforms ``gb_philox_draws`` reads through the device functions the track kernels
call, bit for bit against ``tests/philox.py`` (normals: against a float64 Box-Muller of the same words), and their
distribution.  The tracks: a philox track equals a track fed the same draws as supplied arrays (bit for bit), and the CPU
oracle fed those draws in the reference's order (the free-running assertions of test_gpu_track.py); rows of a track run on
their own with their global point offset (what one rank of a multi-GPU track runs) equal the same rows of the whole track.
"""
import warnings

import numpy as np
import pytest
from scipy import stats

import helpers
import philox
import scenes
from glimpse_b200 import synthetic
from oracle import tracker_oracle as orc

pytestmark = pytest.mark.gpu

SEED = 0x2F4A_1C3B_77E5  # both key words non-zero
SEEDS = [0, 2 ** 32 + 5, 2 ** 62 - 1]
POINTS = [0, 2 ** 31 + 7, 2 ** 32 + 3]
TIMES = [0, 1, 2 ** 31]
# Worst |device float32 Box-Muller - float64 Box-Muller of the same words| seen over the words these tests draw: 7.0e-5, over
# the 12.6 M normals of test_normals_match_a_float64_box_muller on a B200 (1000 W power limit), at a normal of 3.8e-4; asserted
# at twice that.  It is the worst over these words, not a bound on every output: near u = 1 the radius sqrt(-2 ln u) is small and
# badly conditioned.  The word is rounded to float32 first, so words >= 2^32 - 128 give u = 1 and a radius of 0 where the
# float64 radius of the same word is up to 2.4e-4, and words in [2^32 - 256, 2^32 - 129] give u = 1 - 2^-24, where __logf's
# absolute error (2^-21.4) exceeds ln u itself.
NORMAL_ABS_TOL = 1.4e-4


def _lib():
    from glimpse_b200 import _lib as lib

    return lib


# ------------------------------------------------------------------------------------------------ a. the generator
@pytest.mark.parametrize("seed", SEEDS)
def test_generator_bit_for_bit(cuda, seed):
    L = _lib()
    particles = np.append(np.arange(4096, dtype=np.uint64), np.uint64(0xFFFFFFFF))
    worst = 0.0
    for point in POINTS:
        for time in TIMES:
            for stream in range(5):
                got = np.concatenate([philox.read(cuda, L.GB_DRAW_WORDS, seed, point, time, 0, 4096, stream),
                                      philox.read(cuda, L.GB_DRAW_WORDS, seed, point, time, 0xFFFFFFFF, 1, stream)])
                want = philox.words(seed, point, time, particles, stream)
                np.testing.assert_array_equal(got, np.stack(want, axis=1).astype(np.uint32),
                                              err_msg=f"words seed {seed} point {point} time {time} stream {stream}")
                z = np.concatenate([philox.read(cuda, L.GB_DRAW_NORMALS, seed, point, time, 0, 4096, stream),
                                    philox.read(cuda, L.GB_DRAW_NORMALS, seed, point, time, 0xFFFFFFFF, 1, stream)])
                worst = max(worst, float(np.max(np.abs(z - philox.box_muller64(want)))))
            u = philox.read(cuda, L.GB_DRAW_UNIFORM, seed, point, time, 0, 3)
            np.testing.assert_array_equal(u, philox.uniform(seed, point, time + np.arange(3, dtype=np.uint64)))
            up = np.concatenate([philox.read(cuda, L.GB_DRAW_UNIFORM_PARTICLE, seed, point, time, 0, 4096),
                                 philox.read(cuda, L.GB_DRAW_UNIFORM_PARTICLE, seed, point, time, 0xFFFFFFFF, 1)])
            np.testing.assert_array_equal(up, philox.uniform_particle(seed, point, time, particles))
    print("seed", seed, "worst normal error", worst)
    assert worst <= NORMAL_ABS_TOL


def test_normals_match_a_float64_box_muller(cuda):
    """2^21 particles x 2 streams x 3 = 12.6 M device normals against the float64 Box-Muller of the same words: the float32
    construction (__logf, x rsqrt(x), __sincosf of an angle in [0, 2 pi)) stays within NORMAL_ABS_TOL."""
    L = _lib()
    n = 1 << 21
    particles = np.arange(n, dtype=np.uint64)
    worst, where = 0.0, None
    for stream, (point, time) in enumerate([(2 ** 32 + 3, 7), (11, 2 ** 31)]):
        z = philox.read(cuda, L.GB_DRAW_NORMALS, SEED, point, time, 0, n, stream)
        want = philox.box_muller64(philox.words(SEED, point, time, particles, stream))
        err = np.abs(z - want)
        k = int(np.argmax(err))
        if err.flat[k] > worst:
            worst, where = float(err.flat[k]), (stream, k // 3, k % 3, float(want.flat[k]), float(z.flat[k]))
    print("worst |float32 - float64| normal over", 6 * n, "normals:", worst, "(stream, particle, column, float64, device)", where)
    assert worst <= NORMAL_ABS_TOL


# ------------------------------------------------------------------------------------------------ b. the distribution
NORMAL_MOMENTS = {1: (0.0, 1.0), 2: (1.0, 2.0), 3: (0.0, 15.0), 4: (3.0, 96.0)}  # E z^k, Var z^k
UNIFORM_MOMENTS = {1: (0.0, 1 / 12), 2: (1 / 12, 1 / 80 - 1 / 144), 3: (0.0, 1 / 448), 4: (1 / 80, 1 / 2304 - 1 / 6400)}  # of u - 1/2


def assert_moments(x, center, table, label):
    """Mean, variance, skewness and excess kurtosis as the first four moments about the true centre in units of the true
    scale: each sample moment within 5 standard errors of the distribution's."""
    n = x.size
    c = x.ravel() - center
    for k, (mean, var) in table.items():
        m = float(np.mean(c ** k))
        assert abs(m - mean) <= 5 * np.sqrt(var / n), f"{label}: moment {k} = {m}, expected {mean} +- {5 * np.sqrt(var / n)}"


def assert_uncorrelated(a, b, label):
    a, b = a.ravel(), b.ravel()
    r = float(np.corrcoef(a, b)[0, 1])
    assert abs(r) <= 5 / np.sqrt(a.size), f"{label}: correlation {r} over {a.size} pairs"


def test_normals_are_standard_normal(cuda):
    """Device normals over particles 0..2^16-1, four points, three times and streams 0..2 (7.1 M values): moments, KS test
    against N(0,1), and no correlation within a counter, across streams, or between adjacent particles, times and points."""
    L = _lib()
    n = 1 << 16
    points, times = [0, 1, 2 ** 31 + 7, 2 ** 32 + 3], [0, 1, 1000]
    z = np.stack([np.stack([np.stack([philox.read(cuda, L.GB_DRAW_NORMALS, SEED, p, t, 0, n, s) for s in range(3)])
                            for t in times]) for p in points])  # (point, time, stream, particle, 3)
    assert z.size >= 1 << 22
    assert_moments(z, 0.0, NORMAL_MOMENTS, "normals")
    ks = stats.kstest(z.ravel(), "norm")
    print("normals: n", z.size, "KS statistic", ks.statistic, "p", ks.pvalue)
    assert ks.pvalue > 1e-4
    assert_uncorrelated(z[..., 0], z[..., 1], "z0 / z1")
    assert_uncorrelated(z[..., 0], z[..., 2], "z0 / z2")
    assert_uncorrelated(z[..., 1], z[..., 2], "z1 / z2")
    for s0, s1 in ((0, 1), (0, 2), (1, 2)):
        assert_uncorrelated(z[:, :, s0], z[:, :, s1], f"streams {s0} / {s1}")
    assert_uncorrelated(z[:, :, :, 1:], z[:, :, :, :-1], "adjacent particles")
    assert_uncorrelated(z[:, 1], z[:, 0], "adjacent times")
    assert_uncorrelated(z[1], z[0], "adjacent points")


def test_uniforms_are_standard_uniform(cuda):
    """Both uniform kinds (4.2 M values each): moments, KS test against U(0,1), no correlation between adjacent particles,
    times and points."""
    L = _lib()
    n = 1 << 20
    points = [0, 1, 2 ** 32 + 3, 2 ** 32 + 4]
    sysu = np.stack([philox.read(cuda, L.GB_DRAW_UNIFORM, SEED, p, 0, 0, n) for p in points])  # (point, time)
    pu = np.stack([np.stack([philox.read(cuda, L.GB_DRAW_UNIFORM_PARTICLE, SEED, p, t, 0, n // 4) for t in (5, 6, 7, 8)])
                   for p in points])  # (point, time, particle)
    for u, label in ((sysu, "systematic"), (pu, "per particle")):
        assert u.size >= 1 << 22 and u.min() >= 0.0 and u.max() < 1.0
        assert_moments(u, 0.5, UNIFORM_MOMENTS, label)
        ks = stats.kstest(u.ravel(), "uniform")
        print(label, "uniforms: n", u.size, "KS statistic", ks.statistic, "p", ks.pvalue)
        assert ks.pvalue > 1e-4
        assert_uncorrelated(u[1], u[0], f"{label}: adjacent points")
    assert_uncorrelated(sysu[:, 1:], sysu[:, :-1], "systematic: adjacent times")
    assert_uncorrelated(pu[:, 1:], pu[:, :-1], "per particle: adjacent times")
    assert_uncorrelated(pu[..., 1:], pu[..., :-1], "per particle: adjacent particles")


# ------------------------------------------------------------------------------------------------ tracks
class Run:
    """One case set up for the device (a philox Tracker with ``SEED``) and for the oracle."""

    def __init__(self, name):
        import glimpse_b200 as gb
        from glimpse_b200.session import point_span

        self.name = name
        self.scene, self.case = helpers.case_scene(name)
        scene, case = self.scene, self.case
        self.observers, self.models = synthetic.build(scene, gb)
        self.method = case.get("resample_method", "systematic")
        self.cov = bool(case.get("return_covariances", False))
        self.tracker = gb.Tracker(self.observers, seed=SEED, resample_method=self.method,
                                  highpass=case.get("highpass", {"size": (5, 5)}), interpolation=case.get("interpolation", {"kx": 3, "ky": 3}))
        self.tracker._lap = lambda name: None  # (set by track(); _track_local is called directly here)
        matching = self.tracker.match_datetimes(self.tracker.datetimes)
        self.image_index = np.array([[-1 if v is None else int(v) for v in row] for row in matching], dtype=np.int32)
        unit = scene.time_unit.total_seconds()
        self.taus = np.array([dt.total_seconds() / unit for dt in np.diff(self.tracker.datetimes)])
        self.P, self.N = len(self.models), scene.n_particles
        self.mask = np.ones((self.P, len(self.observers)), dtype=bool)
        self.first, self.last = point_span(self.image_index, self.mask)
        self.tangent = np.full(self.P, scene.motion["kind"].startswith("tangent"))
        self.oracle_in = helpers.oracle_inputs(scene)
        np.testing.assert_array_equal(self.oracle_in[3], self.image_index)

    def local(self, lo=0, hi=None, point_offset=None):
        """The device track of rows [lo, hi) alone, keyed from global point ``point_offset`` (default lo)."""
        hi = self.P if hi is None else hi
        return self.tracker._track_local(self.models[lo:hi], self.image_index, self.taus, tuple(self.scene.tile_size),
                                         self.mask[lo:hi], self.cov, True, point_offset=lo if point_offset is None else point_offset,
                                         seed=SEED, n_particles=self.N)

    def draws(self, global_points, lo=0, hi=None):
        hi = self.P if hi is None else hi
        return philox.device_draws(SEED, global_points, self.first[lo:hi], self.last[lo:hi], self.N, self.tangent[lo:hi], self.method)

    def supplied(self, draws):
        """The same track with ``draws`` supplied as arrays (rng_mode = GB_RNG_SUPPLIED), as test_gpu_track.make_session runs it."""
        from glimpse_b200.session import Session

        session = Session(self.tracker, self.models, self.image_index, self.taus, self.scene.tile_size, self.mask,
                          return_covariances=self.cov, return_particles=True, draws=draws)
        session.run()
        return session.fetch()

    def oracle(self, draws, lo=0, hi=None, trace=False):
        """``oracle.tracker_oracle.track`` of rows [lo, hi) fed ``draws`` in the reference's call order."""
        hi = self.P if hi is None else hi
        obs, specs, taus, idx = self.oracle_in
        case = self.case
        r = philox.replay(*draws, steps=self.last[lo:hi] - self.first[lo:hi], tangent=self.tangent[lo:hi], method=self.method)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            res = orc.track(obs, specs[lo:hi], taus, idx, tile_size=self.scene.tile_size, return_particles=True,
                            return_covariances=self.cov, randn=r.randn, random=r.random, resample_method=self.method,
                            highpass_size=case.get("highpass", {"size": (5, 5)}).get("size"),
                            highpass_kwargs={k: v for k, v in case.get("highpass", {}).items() if k != "size"},
                            raise_errors=True, trace=trace, **case.get("interpolation", {}))
        assert r.done, "the oracle left device draws unused"
        return res


# Cases where, with the draws of SEED, one point's ancestors differ from the oracle's from some update on (measured on a B200:
# track_hp_nearest point 0 at time 4, track_jitter point 0 at time 3, shape_c2 point 0 at its first update), the means agreeing
# to 2e-7 sigma before it.  At that update test_philox_track_matches_the_oracle forces the oracle's evolved particles into the
# step and requires a near-tie (assert_near_ties): device weights within the teacher-forced tolerance of the oracle's, and every
# child whose ancestor differs has its resampling position between the oracle's and the device's cumulative weight at the
# boundary it crossed.  After that update they get the shape-case (statistical) assertions.
ANCESTOR_FLIPS = {"track_hp_nearest", "track_jitter", "shape_c2"}
WEIGHT_REL = 3e-4  # device vs reference weights of one update (test_gpu_track.test_step_teacher_forced)


def assert_matches_oracle(run, means, sig, particles, res):
    """The assertions of test_gpu_track.test_track_free_running_matches_reference against the oracle's result ``res``: exact
    agreement (1e-5) at every time before each point's first differing ancestor; after it, none allowed (small cases) or
    statistical agreement (shape cases and ANCESTOR_FLIPS).  Returns the first differing time of every point (T: none)."""
    name = run.name
    same = np.isclose(particles, res.particles, rtol=0, atol=1e-9).all(axis=3)  # (P, T, N)
    frac = 1.0 - same.mean()
    sig_ref = res.sigmas if not run.cov else np.sqrt(np.einsum("ptii->pti", res.sigmas))
    d = np.abs(means - res.means) / np.maximum(sig_ref, 1e-12)
    d = d[..., [0, 1, 3, 4]] if name not in ("track_cyl2", "shape_c3") else d
    T = same.shape[1]
    diverged = ~same.all(axis=2)
    first_div = np.where(diverged.any(axis=1), diverged.argmax(axis=1), T)
    before = np.arange(T)[None, :] < first_div[:, None]
    d_before = np.nanmax(np.where(before[..., None], d, 0.0))
    print(name, "particle mismatch fraction", frac, "max |dmean|/sigma", np.nanmax(d), "before the first differing ancestor", d_before,
          "first differing time per point", first_div.tolist())
    assert d_before <= 1e-5
    if not run.cov:
        ok = (res.sigmas > 0) & before[..., None]
        assert np.max(np.abs(sig[ok] - res.sigmas[ok]) / res.sigmas[ok], initial=0.0) <= 1e-5
    if name in scenes.shape_cases() or name in ANCESTOR_FLIPS:
        assert np.nanmax(d) < 0.5 and np.nanmedian(d) < 0.02
        if run.N <= 10000 and name not in ANCESTOR_FLIPS:
            assert first_div.min() >= 2
        if not run.cov:
            ok = res.sigmas > 0
            assert np.nanmedian(np.abs(sig[ok] - res.sigmas[ok]) / res.sigmas[ok]) < 0.02
        return first_div
    assert frac <= 1e-4
    assert np.nanmax(d) <= 1e-5
    if not run.cov:
        ok = res.sigmas > 0
        assert np.nanmax(np.abs(sig[ok] - res.sigmas[ok]) / res.sigmas[ok]) <= 1e-5
    return first_div


def resample_positions(method, u, N):
    """The points the reference's resamplers search in the normalised cumulative weights (oracle systematic_indices,
    stratified_indices, choice_indices)."""
    if method in ("systematic", "stratified"):
        return (np.arange(N) + np.asarray(u)) * (1 / N)
    assert method == "choice", method
    return np.asarray(u)


def assert_near_ties(run, draws, res, first_div, differs):
    """At each point's first differing update (``first_div``, from a run of the oracle with ``trace=True``), the device step
    with the oracle's evolved particles forced in: its weights are within WEIGHT_REL of the oracle's; the children whose
    ancestor differs include every child that differs in the free-running track there (``differs[p]``); and each of them
    moved by one parent across a boundary b with its position between the oracle's and the device's normalised cumulative
    weight at b — a near-tie decided by the measured weight noise, not a wrong ancestor.  (The device sums the cumulative
    weights in its own order: 1e-12 of slack.)"""
    import torch

    from glimpse_b200 import _lib as L
    from glimpse_b200.session import Session

    P, N, T = run.P, run.N, res.means.shape[1]
    steps = {(s["p"], s["t"]): s for s in res.trace if "indices" in s}
    session = Session(run.tracker, run.models, run.image_index, run.taus, run.scene.tile_size, run.mask,
                      return_covariances=run.cov, return_particles=True, draws=draws)
    session.run()  # (the templates)
    torch.cuda.synchronize()
    dev = session.device
    for p in np.nonzero(first_div < T)[0]:
        t = int(first_div[p])
        s = steps[(p, t)]
        evolved = np.stack([steps[(q, t)]["evolved"] if (q, t) in steps else np.zeros((N, 6)) for q in range(P)])
        f_ev = torch.as_tensor(np.ascontiguousarray(evolved.transpose(0, 2, 1))).to(dev)  # (P, 6, N)
        w_dump = torch.zeros((P, N), dtype=torch.float64, device=dev)
        i_dump = torch.full((P, N), -1, dtype=torch.int32, device=dev)
        io = L.gb_stage_io()
        io.force_evolved, io.dump_weights, io.dump_indices = f_ev.data_ptr(), w_dump.data_ptr(), i_dump.data_ptr()
        session.buf["status"].zero_()
        session.step(t, io)
        torch.cuda.synchronize()
        w_d, k_d = w_dump[p].cpu().numpy(), i_dump[p].cpu().numpy().astype(np.int64)
        w_o, k_o = s["weights"], np.asarray(s["indices"])
        rel = float(np.max(np.abs(w_d - w_o) / w_o))
        assert rel <= WEIGHT_REL, f"point {p} time {t}: weights {rel} from the oracle's"
        c_o, c_d = np.cumsum(w_o / w_o.sum()), np.cumsum(w_d / w_d.sum())
        if run.method == "choice":
            c_o, c_d = c_o / c_o[-1], c_d / c_d[-1]
        pos = resample_positions(run.method, s["u"], N)
        flipped = np.nonzero(k_d != k_o)[0]
        assert set(differs[p].tolist()) <= set(flipped.tolist()), (p, t, differs[p], flipped)
        b = np.minimum(k_d[flipped], k_o[flipped])
        assert np.all(np.abs(k_d[flipped] - k_o[flipped]) == 1), (k_d[flipped], k_o[flipped])
        gap, noise = np.abs(pos[flipped] - c_o[b]), np.abs(c_d[b] - c_o[b])
        print(run.name, "point", p, "time", t, "weights within", rel, "of the oracle's;", len(flipped), "ancestors differ; their",
              "position - boundary", gap.tolist(), "cumulative-weight difference at the boundary", noise.tolist())
        between = (pos[flipped] >= np.minimum(c_o[b], c_d[b]) - 1e-12) & (pos[flipped] <= np.maximum(c_o[b], c_d[b]) + 1e-12)
        assert between.all() and np.all(gap <= noise + 1e-12), "an ancestor differs beyond the measured weight noise"


CASES = list(scenes.track_cases())
RESULT_KEYS = ("means", "sigmas", "status", "status_time", "obs_flags", "particles", "weights")


@pytest.mark.parametrize("name", CASES)
def test_philox_track_equals_supplied_draw_track(cuda, name):
    """c. rng_mode only selects where the draws come from: the philox track and the track given the device's draws as
    arrays are identical."""
    run = Run(name)
    mine = run.local()
    assert (mine["status"] == 0).all(), mine["status"]
    given = run.supplied(run.draws(range(run.P)))
    for key in RESULT_KEYS:
        np.testing.assert_array_equal(mine[key], given[key], err_msg=f"{name}: {key}")


@pytest.mark.parametrize("name", CASES + ["shape_c1", "shape_c2"])
def test_philox_track_matches_the_oracle(cuda, name):
    """d. Tracker.track with the device draws against the oracle fed the same draws."""
    run = Run(name)
    tracks = run.tracker.track(run.models, tile_size=run.scene.tile_size, return_particles=True, return_covariances=run.cov)
    assert all(e is None for e in tracks.errors)
    draws = run.draws(range(run.P))
    res = run.oracle(draws, trace=name in ANCESTOR_FLIPS)
    first_div = assert_matches_oracle(run, tracks.means, tracks.covariances if run.cov else tracks.sigmas, tracks.particles, res)
    if name in ANCESTOR_FLIPS:
        T = res.means.shape[1]
        same = np.isclose(tracks.particles, res.particles, rtol=0, atol=1e-9).all(axis=3)
        differs = [np.nonzero(~same[p, first_div[p]])[0] if first_div[p] < T else None for p in range(run.P)]
        assert_near_ties(run, draws, res, first_div, differs)


@pytest.mark.parametrize("name,lo,hi", [("track_c1", 1, 3), ("track_c1", 2, 3), ("track_residual", 1, 2), ("track_choice", 1, 2),
                                        ("track_tangent", 1, 2), ("track_cyl2", 1, 2)])
def test_rows_keyed_by_their_global_point_index(cuda, name, lo, hi):
    """e. Rows [lo, hi) run alone with point_offset = lo (what one rank of a multi-GPU track runs) equal those rows of the
    whole track and the oracle fed the draws of global points lo ... hi - 1."""
    run = Run(name)
    whole = run.local()
    part = run.local(lo, hi)
    for key in RESULT_KEYS:
        np.testing.assert_array_equal(part[key], whole[key][lo:hi], err_msg=f"{name} rows [{lo}, {hi}): {key}")
    res = run.oracle(run.draws(range(lo, hi), lo, hi), lo, hi)
    assert_matches_oracle(run, part["means"], part["sigmas"], part["particles"], res)


@pytest.mark.parametrize("name", ["track_c1", "track_stratified"])
def test_point_offset_beyond_32_bits(cuda, name):
    """e. A block of points keyed from global point 2^32 + 1 (the high point word of the counter) against the oracle fed the
    draws of those global points."""
    run = Run(name)
    offset = 2 ** 32 + 1
    mine = run.local(point_offset=offset)
    assert (mine["status"] == 0).all()
    assert not np.array_equal(mine["means"], run.local()["means"])
    res = run.oracle(run.draws(range(offset, offset + run.P)))
    assert_matches_oracle(run, mine["means"], mine["sigmas"], mine["particles"], res)
