"""Float64 replay of every update of a track from the track's own outputs.

A ``gb_track`` run with ``return_particles=True`` returns, for every point p and time t, the resampled particles
``particles[p, t]``, the weights they carry ``weights[p, t]``, the moments, ``obs_flags`` and (through the session) the
realised search-window sizes.  Given the outputs at t - 1 and the draws of t, update t is determined: the replay evolves
``particles[p, t - 1]`` with the oracle's motion step, computes the pre-resample weights (carried, uniform, DEM-only or
through the oracle's closed-form tile pipeline), resamples with the oracle's ``systematic_indices`` /
``stratified_indices`` (the pipelined flow) or ``choice_indices`` / ``residual_indices`` (the step-by-step flow), and checks
the device's update against it.  Each update starts from the device's own previous
outputs, so one flipped ancestor does not make the rest of the track diverge: every update is checked on its own.

What ``replay_track`` asserts, per update:
* propagation: every child row equals exactly one row of the evolved particles (rtol = atol = 1e-13, the tolerance of
  ``test_stand_alone_evolve_particles_matches_the_oracle``; the second nearest row is far outside it), which recovers the
  device's ancestors; at the first time the particles equal ``init_particles`` of the init draws and the weights are 1;
* structure: children of one parent bitwise-equal rows with bitwise-equal weights; ancestors non-decreasing (systematic,
  stratified; choice children are in draw order, residual ones repetitions first);
* weights: carried and uniform updates bit for bit (``w_pre[k]``); DEM-only within ``DEM_REL`` (the ``exp_neg_fast``
  bound); observed within ``WEIGHT_REL``;
* ancestors: equal to the reference's, or a near-tie: moved across one boundary b of the cumulative weights C (by one
  parent, or over parents whose weights add up to no more than the band) with |pos - C[b]| <= delta min(C[b], 1 - C[b]) + 1e-12, delta = 0 at carried / uniform updates, 2 DEM_REL at DEM-only ones,
  2 WEIGHT_REL at observed ones; choice: the position is the child's uniform, C is normalised by C[-1];
  residual (``check_residual``): bit-equal at carried / uniform updates; elsewhere the device's repetitions within the weight
  noise of floor(N wn) and every additional child an answer NumPy's search can reach, comparisons within the noise going
  either way;
* moments: means, sigmas or covariances against a long-double reference of the device's own particles and weights, taken
  about particle 0 (means 1e-9 sigma, variances 2e-7 relative, covariances 1e-7 sqrt(c_ii c_jj), plus two float64 ulps of
  the value for the rounding of the stored result).  The device sums one pass of first and second moments about the
  point's moment origin r, fixed by k_init from the prior (xy, the DEM there, the prior velocity: ``moment_origin``), so
  var = E[d^2] - E[d]^2 with d = x - r, whose rounding is a few eps max d^2: 16 eps D_i D_j is allowed on top, D = the
  largest |x - r| of the particles.  It matters only where the spread has collapsed far below the distance from r (two
  children of one parent at N = 2: sigma 2e-9 m where the reference has 0);
* next window: ``obs_flags`` equal the oracle's skip codes, and the width and height of every used window equal those of
  the oracle's ``search_window`` of the evolved particles (+-1 in the width only where an unrounded left or right edge lies
  within 1e-9 px of an integer, in the height likewise for the top or bottom edge; such cases are counted).
"""
import numpy as np
from scipy.spatial import cKDTree

import helpers
from oracle import tracker_oracle as orc

WEIGHT_REL = 3e-4  # observed updates: device vs reference weights (test_gpu_track.test_step_teacher_forced)
DEM_REL = 3e-7     # DEM-only updates: exp_neg_fast's relative error (DESIGN §5 "Weights")
PROP_TOL = 1e-13   # motion step: rtol = atol
SEED = 0x5EED_0F_A11  # the philox key of the GPU replay (the host coverage test restates its draws)
KINDS = ("carried", "uniform", "dem", "observed")
CHUNK = 768        # children per k_s4p chunk / particles per block at most
EPS = np.finfo(float).eps
STEP_METHODS = ("choice", "residual")  # resamplers of the step-by-step flow


# ------------------------------------------------------------------------------------------------ scenes
def interleave(scene, offset_hours=12):
    """Add an observer holding copies of the first observer's frames at datetimes ``offset_hours`` later: with it masked
    out, a point has times without any image (``parse_datetimes`` would drop such times from a plain ``datetimes=``)."""
    import datetime

    from glimpse_b200 import synthetic

    o = scene.observers[0]
    dt = datetime.timedelta(hours=offset_hours)
    scene.observers.append(synthetic.ObserverScene([f.copy() for f in o.frames], np.array(o.cams, copy=True),
                                                   [d + dt for d in o.datetimes], o.sigma))
    return scene


def fine_dem_sigma(scene, cells=(140, 180), lo=0.01, hi=0.05):
    """The gridded DEM of ``scenes.add_gridded_dem`` with a DEM sigma of 0.5 m cells between ``lo`` and ``hi`` m."""
    import scenes

    scenes.add_gridded_dem(scene)
    rng = np.random.RandomState(12)
    dem = scene.motion["dem"]
    scene.motion["dem_sigma"] = dict(array=lo + (hi - lo) * rng.rand(*cells), x=dem["x"], y=dem["y"])
    return scene


def stream_block(N):
    """gb_step_plan's particles per block for N particles: CHUNK at most, even, as equal as possible."""
    nblk = -(-N // CHUNK)
    return (-(-N // nblk) + 1) // 2 * 2


def case(name, n_particles=None, method=None):
    """(scene, observer mask, resample method, covariances) of a replay case: every case has an interleaved observer (the
    last one) that the mask takes away from some points, so that they take updates without any image.  ``n_particles``
    overrides the case's particle count (host tests of the replay itself), ``method`` its resampler.  ``scene.meta["kinds"]`` = the motion kind of
    every point where they differ, ``scene.meta["reverse"]`` = the track runs its datetimes backwards (``build``,
    ``inputs``, ``datetimes``)."""
    import scenes
    from glimpse_b200 import synthetic

    small = dict(imgsz=(320, 240), margin_px=100)
    case_method, cov, later, kinds, reverse = "systematic", False, None, None, False
    if name == "tan_carried_collapse":
        scene = synthetic.nadir_scene(seed=61, n_points=1, n_particles=100000, n_frames=3, kind="tangent_cartesian", **small)
        scenes.add_gridded_dem(scene)
        scene.observers[0].sigma = 0.007  # weights collapse onto a few parents at the observed updates
        masked = [0]
    elif name == "tan_cyl_stratified_odd":
        scene = synthetic.nadir_scene(seed=62, n_points=2, n_particles=9999, n_frames=3, kind="tangent_cylindrical",
                                      velocity_sigma=0.2, **small)
        scenes.add_gridded_dem(scene)
        case_method, cov, masked = "stratified", True, [0]
        later = 1  # sees the interleaved observer only: starts half a time unit after point 0
    elif name == "cart_dem_floor":
        scene = synthetic.nadir_scene(seed=63, n_points=2, n_particles=10000, n_frames=3, **small)
        fine_dem_sigma(scene)
        scene.motion["vxyz_sigma"] = (0.3, 0.3, 0.5)  # log-likelihoods of 0 .. ~1000 half a day after the first frame
        masked = [0, 1]
    elif name == "shape_c2_interleaved":
        _, c = helpers.case_scene("shape_c2")
        scene = synthetic.nadir_scene(**dict(c["scene_kwargs"], n_frames=4))
        masked = [0]
    elif name == "million":
        scene = synthetic.nadir_scene(seed=64, n_points=1, n_particles=1000001, n_frames=2, kind="tangent_cartesian", **small)
        scenes.add_gridded_dem(scene)
        masked = [0]
    elif name == "mixed_three_obs":
        # three observers (the second rolled by 180 deg, RGB, from the second frame on; the interleaved one): k_s4p projects
        # into observer slot 2 through its generic loop.  Cartesian, cylindrical and tangent points in one call, datetimes
        # backwards (tau < 0).  Point 1's template box leaves the frame at its first time: it fails inside a batch of active
        # points.  Points 0, 2 and 3 do not see the interleaved observer, so they start at t = 1 (the last frame of the first
        # observer, the track running backwards) and take uniform, DEM-only and carried updates.
        scene = synthetic.nadir_scene(seed=67, n_points=4, n_particles=2000, n_frames=3, **small)
        scenes.add_second_observer(scene)
        scene.points = np.insert(scene.points, 1, [(3 - 160) * 0.2, 0.0], axis=0)
        kinds = ["cartesian", "cartesian", "cylindrical", "tangent_cartesian", "tangent_cartesian"]
        masked, reverse = [0, 2, 3], True
    elif name.startswith("small_"):  # small_<N>
        scene = synthetic.nadir_scene(seed=65, n_points=2, n_particles=int(name[6:]), n_frames=3, **small)
        # a point between them whose template box leaves the frame: it fails at its first time, the others carry on
        scene.points = np.insert(scene.points, 1, [(3 - 160) * 0.2, 0.0], axis=0)
        masked = [0]
    else:
        raise KeyError(name)
    if n_particles is not None:
        scene.n_particles = int(n_particles)
    method = method or case_method
    scene.meta.update(kinds=kinds, reverse=reverse)
    interleave(scene)
    P, O = len(scene.points), len(scene.observers)
    mask = np.ones((P, O), dtype=bool)
    mask[masked, O - 1] = False
    if later is not None:
        mask[later, :O - 1] = False
    return scene, mask, method, cov


CASES = ["tan_carried_collapse", "tan_cyl_stratified_odd", "cart_dem_floor", "shape_c2_interleaved", "mixed_three_obs", "million",
         "small_2", "small_37", "small_769"]
# the step-by-step flow (k_s1_propagate -> k_s2 -> k_s3 -> k_s4c_scan or k_s4r_residual -> k_s4c_gather -> k_s5_finalize):
# (case, resampler); small_99005 takes uniform updates at N (1 / N) < 1, where the residual resampler has no repetitions
STEP_CASES = [("tan_carried_collapse", "choice"), ("million", "choice"), ("mixed_three_obs", "choice"),
              ("tan_cyl_stratified_odd", "residual"), ("cart_dem_floor", "residual"), ("small_99005", "residual")]


def _kind_scene(scene, kind):
    """``scene`` with the motion parameters ``synthetic.nadir_scene`` gives ``kind`` (the default drift and spreads)."""
    import copy

    from glimpse_b200 import synthetic

    out = copy.copy(scene)
    out.motion = synthetic.nadir_scene(seed=0, n_points=1, n_particles=1, n_frames=1, imgsz=(64, 48), margin_px=10, kind=kind).motion
    return out


def build(scene, api):
    """(observers, motion models) of a replay case for ``api`` (this package), one model per point of its own kind."""
    from glimpse_b200 import synthetic

    observers, models = synthetic.build(scene, api)
    kinds = scene.meta.get("kinds")
    if kinds is not None:
        models = [synthetic.build(_kind_scene(scene, k), api, points=[i])[1][0] for i, k in enumerate(kinds)]
    return observers, models


def inputs(scene):
    """``helpers.oracle_inputs`` of a replay case, with one MotionSpec per point of its own kind and, for a backward track,
    the times in the order the track runs them (image_index reversed, taus negative)."""
    observers, specs, taus, image_index = helpers.oracle_inputs(scene)
    kinds = scene.meta.get("kinds")
    if kinds is not None:
        specs = [helpers.oracle_inputs(_kind_scene(scene, k), points=[i])[1][0] for i, k in enumerate(kinds)]
    if scene.meta.get("reverse"):
        image_index, taus = image_index[::-1].copy(), -taus[::-1]
    return observers, specs, taus, image_index


def datetimes(scene):
    """The ``datetimes`` argument of the case's ``Tracker.track`` call (None: the observers' own, ascending)."""
    return scene.datetimes[::-1] if scene.meta.get("reverse") else None


def update_kinds(specs, image_index, mask):
    """Kind of every update (p, t > first[p]) from the scene alone: 'observed' where an observer the point sees has an image,
    otherwise 'carried' (tangent models), 'uniform' (DEM sigma identically 0) or 'dem'.  Returns {(p, t): kind}."""
    out = {}
    for p, m in enumerate(specs):
        seen = (image_index[:, mask[p]] >= 0).any(axis=1)
        first, last = int(np.argmax(seen)), len(seen) - 1 - int(np.argmax(seen[::-1]))
        for t in range(first + 1, last + 1):
            if seen[t]:
                out[(p, t)] = "observed"
            elif m.tangent:
                out[(p, t)] = "carried"
            elif not np.any(m.dem_sigma.array):
                out[(p, t)] = "uniform"
            else:
                out[(p, t)] = "dem"
    return out


# ------------------------------------------------------------------------------------------------ draws
def feeder(*blocks):
    """``randn`` handing out ``blocks`` in order (shape-checked)."""
    queue = list(blocks)

    def randn(*shape):
        value = queue.pop(0)
        assert value.shape == tuple(shape), (value.shape, shape)
        return np.array(value)

    return randn


def init_draws(init, tangent):
    return feeder(init[:, 0:2], init[:, 2], init[:, 3:5] if tangent else init[:, 3:6])


def step_draws(step, tangent):
    return feeder(step[:, 0:2], step[:, 2]) if tangent else feeder(step)


def random_draws(n, seed):
    """Draws in the layout of ``philox.device_draws`` from NumPy's generator (host tests)."""
    rng = np.random.RandomState(seed)
    return rng.randn(*n[0]), rng.randn(*n[1]), rng.random_sample(n[2])


# ------------------------------------------------------------------------------------------------ the replay
def window_edges(uv, size, kx, ky):
    """``orc.search_window``'s box before floor / ceil."""
    size = np.asarray(size)
    half = size * 0.5
    box = np.vstack((uv.min(axis=0) - half, uv.max(axis=0) + half))
    ncols = ky - ((box[1, 0] - box[0, 0]) - size[0])
    if ncols > 0:
        box[:, 0] += np.array((-ncols, ncols)) * 0.5
    nrows = kx - ((box[1, 1] - box[0, 1]) - size[1])
    if nrows > 0:
        box[:, 1] += np.array((-nrows, nrows)) * 0.5
    return box.ravel()


def moments_ref(ps, w, cov):
    """Weighted mean and sigmas (or covariance) of ``ps`` in long double, about particle 0."""
    ld = np.longdouble
    d = ps.astype(ld) - ps[0].astype(ld)
    wl = w.astype(ld)
    W = wl.sum()
    m1 = (wl[:, None] * d).sum(axis=0) / W
    c = d - m1
    mean = ps[0].astype(ld) + m1
    if cov:
        return mean, (wl[:, None, None] * c[:, :, None] * c[:, None, :]).sum(axis=0) / W
    return mean, np.sqrt((wl[:, None] * c * c).sum(axis=0) / W)


def recover_ancestors(children, evolved):
    """Index of the evolved row every child equals (to PROP_TOL), and the worst error |child - row| / (1 + |row|); the
    nearest row must be within the tolerance and the second nearest far outside it."""
    scale = PROP_TOL * (1 + np.abs(evolved).max(axis=0))
    tree = cKDTree(evolved / scale)
    k = min(2, len(evolved))
    dist, idx = tree.query(children / scale, k=k, p=np.inf)
    dist, idx = dist.reshape(len(children), k), idx.reshape(len(children), k)
    anc = idx[:, 0]
    err = np.abs(children - evolved[anc])
    bound = PROP_TOL * (1 + np.abs(evolved[anc]))
    bad = np.nonzero(~(err <= bound).all(axis=1))[0]
    assert len(bad) == 0, f"child {bad[:5].tolist()} matches no evolved particle (nearest at {dist[bad[:5], 0].tolist()} tolerances)"
    if k == 2:
        close = np.nonzero(dist[:, 1] <= 1e3)[0]
        assert len(close) == 0, f"child {close[:5].tolist()} matches two evolved particles"
    return anc.astype(np.int64), float((err / (1 + np.abs(evolved[anc]))).max())


class Report(dict):
    def worst(self, key, value):
        self[key] = max(self.get(key, 0.0), float(value))

    def count(self, key, n=1):
        self[key] = self.get(key, 0) + int(n)


def moment_origin(spec):
    """The moment origin k_init stores for a point (glimpse_b200.cu, k_init): the prior xy, the DEM there (0 if NaN), the
    prior velocity (a cylindrical model's as vx, vy; the other models' first two components as given), v[2]."""
    xy = np.asarray(spec.xy, dtype=float)
    z = float(spec.dem.sample(xy[None, :])[0])
    v = np.asarray(spec.v, dtype=float)
    vxy = (v[0] * np.cos(v[1]), v[0] * np.sin(v[1])) if spec.kind == "cylindrical" else (v[0], v[1])
    return np.array([xy[0], xy[1], 0.0 if np.isnan(z) else z, vxy[0], vxy[1], v[2]])


def check_moments(rep, res, p, t, cov, tag, origin, terms=None):
    """``terms``: a one-pass allowance of terms eps D on the means and terms eps D_i D_j on the (co)variances, for sums over a
    chain of up to ``terms`` additions taken far from a collapsed cloud (test_gpu_resample_step).  None: the replay's own
    allowance, 16 eps D_i D_j on the (co)variances and none on the means."""
    ps, w = res["particles"][p, t], res["weights"][p, t]
    mean, sig = moments_ref(ps, w, cov)
    got_m, got_s = res["means"][p, t], res["sigmas"][p, t]
    s = np.sqrt(np.diagonal(sig).astype(float)) if cov else sig.astype(float)
    mean = mean.astype(float)
    dm = np.abs(got_m - mean)
    ulp = lambda x: 2 * np.spacing(np.abs(x))  # noqa: E731
    step = np.abs(ps - origin).max(axis=0)
    # the mean is r + E[d]: where the spread has collapsed the rounding of E[d], terms eps D, is all that is left
    mean_pass = 0.0 if terms is None else terms * EPS * step
    assert (dm <= 1e-9 * s + ulp(mean) + mean_pass).all(), f"{tag}: means {got_m} against {mean} (sigma {s})"
    spread = s > 1e-7 * step  # (relative errors are reported where the spread has not collapsed)
    rep.worst("mean/sigma", np.max(np.where(spread, dm / np.where(spread, s, 1), 0)))
    rep.worst("mean abs where the spread collapsed", np.max(np.where(spread, 0, dm)))
    one_pass = (16 if terms is None else terms) * EPS * np.outer(step, step)
    if cov:
        c = sig.astype(float)
        scale = np.sqrt(np.outer(s, s))
        dc = np.abs(got_s - c)
        assert (dc <= 1e-7 * scale + one_pass + ulp(c)).all(), \
            f"{tag}: covariances off by {np.max(dc / np.maximum(scale, 1e-300))} of sqrt(c_ii c_jj)"
        both = np.outer(spread, spread)
        rep.worst("cov rel", np.max(np.where(both, dc / np.where(both, scale, 1), 0)))
    else:
        dv = np.abs(got_s ** 2 - s ** 2)
        assert (dv <= 2e-7 * s ** 2 + np.diagonal(one_pass) + ulp(s ** 2)).all(), f"{tag}: sigmas {got_s} against {s}"
        rep.worst("sigma rel", np.max(np.where(spread, np.abs(got_s - s) / np.where(spread, s, 1), 0)))
        rep.worst("sigma abs where the spread collapsed", np.max(np.where(spread, 0, np.abs(got_s - s))))


def check_near_ties(rep, anc, idx, w_pre, pos, delta, kind, tag, choice=False):
    """The device's ancestors ``anc`` against the reference's ``idx``: equal, or a near-tie — moved across one boundary b of
    the normalised cumulative weights C (by one parent, or over parents whose weights add up to no more than the band), the
    child's position ``pos`` within delta min(C[b], 1 - C[b]) of C[b], plus the rounding of two summation orders of C (1e-12;
    choice: C is normalised by C[-1] and divides the device's block-wise sums by their total, (N + 2) eps C at least).
    Returns the differing children."""
    flipped = np.nonzero(anc != idx)[0]
    if len(flipped):
        N = len(w_pre)
        C = np.cumsum(w_pre / w_pre.sum())
        if choice:
            C /= C[-1]
        a, b = np.minimum(anc[flipped], idx[flipped]), np.maximum(anc[flipped], idx[flipped])
        slack = np.maximum(1e-12, (N + 2) * EPS * C[b - 1]) if choice else 1e-12
        band = delta * np.minimum(C[a], 1 - C[a]) + slack
        between = C[b - 1] - C[a]  # weight of the parents strictly between the two: inside the weight noise
        assert (between <= band).all(), \
            f"{tag}: children {flipped[:5].tolist()} have ancestors {anc[flipped[:5]].tolist()}, reference {idx[flipped[:5]].tolist()}"
        pos = pos[flipped] if np.ndim(pos) else pos
        gap = np.abs(pos - C[a])
        assert (gap <= band).all(), \
            f"{tag}: ancestors of children {flipped[:5].tolist()} differ beyond a near-tie (gaps {gap[:5].tolist()})"
        print(f"{tag}: {len(flipped)} near-ties at a {kind} update, |position - boundary| {gap.max():.3g}, "
              f"most parents crossed {int((b - a).max())}")
    return flipped


def searchsorted_reachable(cs, key, lo, hi, band):
    """The answers np.searchsorted's binary search (side 'left', from the bounds [lo, hi)) can reach on ``cs`` when every
    comparison with |cs[mid] - key| <= band may go either way."""
    out, todo, seen = set(), [(lo, hi)], set()
    while todo:
        lo, hi = todo.pop()
        if (lo, hi) in seen:
            continue
        seen.add((lo, hi))
        if lo >= hi:
            out.add(lo)
            continue
        mid = lo + ((hi - lo) >> 1)
        d = cs[mid] - key
        if d < 0 or abs(d) <= band:
            todo.append((mid + 1, hi))
        if d >= 0 or abs(d) <= band:
            todo.append((lo, mid))
    return out


def carried_bounds(keys, prev, N):
    """NumPy's search bounds (numpy/_core/src/npysort/binsearch.cpp) for each key after the previous key's search ended at
    ``prev`` (its state is its answer): [prev, N) after a smaller key, else [0, min(prev + 1, N)).  The first key: [0, N)."""
    lo, hi = np.zeros(len(keys), dtype=np.int64), np.full(len(keys), N, dtype=np.int64)
    if len(keys) > 1:
        up = keys[:-1] < keys[1:]
        lo[1:] = np.where(up, prev, 0)
        hi[1:] = np.where(up, N, np.minimum(prev + 1, N))
    return lo, hi


def check_residual(rep, anc, w_pre, row, delta, kind, tag):
    """The residual resampler's ancestors (oracle.residual_indices: repetitions of floor(N wn), then np.searchsorted of the
    uniforms ``row[:N - K]`` on the cumulative sum of wn - repetitions).  Exact weights (delta = 0): bit-equal to the
    reference's.  Otherwise the repetitions may differ where the weight noise moves N wn across an integer: the device's K is
    found among the last few children of the ancestors' longest non-decreasing prefix, its repetitions bincount(anc[:K]) must
    lie within floor(N wn (1 -+ delta)), and every additional child must be an answer NumPy's search can reach on the
    cumulative sum rebuilt from the reference's wn and those repetitions, starting from the device's previous answer, when
    comparisons within the noise of that sum may go either way."""
    N = len(w_pre)
    if delta == 0:
        ref, used = orc.residual_indices(w_pre, lambda m: row[:m])
        bad = np.nonzero(anc != ref)[0]
        assert len(bad) == 0, \
            f"{tag}: K {N - len(used)}, children {bad[:5].tolist()} have ancestors {anc[bad[:5]].tolist()}, reference {ref[bad[:5]].tolist()}"
        rep.count(f"residual K = 0 ({kind})", len(used) == N)
        return
    wn = w_pre / w_pre.sum()
    reps_lo, reps_hi = np.floor(N * wn * (1 - delta)), np.floor(N * wn * (1 + delta))
    dec = np.nonzero(np.diff(anc) < 0)[0]
    prefix = int(dec[0]) + 1 if len(dec) else N
    why = "no K satisfies the repetition bounds"
    for K in range(prefix, max(prefix - 8, 0) - 1, -1):
        reps = np.bincount(anc[:K], minlength=N)
        if not ((reps_lo <= reps) & (reps <= reps_hi)).all():
            continue
        residuals = wn - reps
        residuals *= 1 / residuals.sum()
        cs = np.cumsum(residuals)
        cs[-1] = 1.0
        keys, got = row[:N - K], anc[K:]
        # wn carries up to delta of relative error (tol in the weights, tol in their sum), so |d cs| <= delta (1 + |cs|) / |1 - K|
        # (the residuals sum to 1 - K), plus the rounding of the sums
        band = delta * (1 + np.abs(cs).max()) / max(abs(1 - K), 1) + (N + 2) * EPS * np.abs(cs).max()
        lo, hi = carried_bounds(keys, got[:-1], N)
        lo0, hi0 = lo.copy(), hi.copy()
        while (lo < hi).any():  # the exact search from the device's state, every key at once
            mid = lo + ((hi - lo) >> 1)
            go = cs[np.minimum(mid, N - 1)] < keys
            lo, hi = np.where((lo < hi) & go, mid + 1, lo), np.where((lo < hi) & ~go, mid, hi)
        off = np.nonzero(lo != got)[0]
        if all(int(got[i]) in searchsorted_reachable(cs, keys[i], int(lo0[i]), int(hi0[i]), band) for i in off):
            rep.worst(f"residual repetitions off floor(N wn) ({kind})", np.abs(reps - np.floor(N * wn)).max(initial=0))
            rep.count(f"residual searches within the noise ({kind})", len(off))
            return
        why = f"K {K}: additional children {off[:5].tolist()} unreachable"
    raise AssertionError(f"{tag}: residual ancestors: {why} (non-decreasing prefix {prefix})")


def replay_track(res, draws, scene_inputs, method, mask, tile_size, cov=False, windows=None, highpass_size=(5, 5), kx=3, ky=3):
    """Replay every update of every point of the track ``res`` (dict: means, sigmas, particles, weights, obs_flags, status,
    status_time) taken with ``draws`` = (init, step, unif) in the layout of ``philox.device_draws``.  ``scene_inputs`` =
    ``helpers.oracle_inputs`` (one MotionSpec per point), ``windows`` = the session's (P, T, O, 2) window sizes or None.
    A failed point is replayed up to its failure, where the replay must fail too.  Raises AssertionError at the first
    difference; returns a Report of worst values and counts."""
    observers, specs, taus, image_index = scene_inputs
    init, step, unif = draws
    P, T, O = res["obs_flags"].shape
    template_frame = np.array([int(np.argmax(image_index[:, o] >= 0)) for o in range(O)])
    rep = Report()
    for p, model in enumerate(specs):
        seen = (image_index[:, mask[p]] >= 0).any(axis=1)
        first, last = int(np.argmax(seen)), len(seen) - 1 - int(np.argmax(seen[::-1]))
        failed = int(res["status"][p]) != 0
        stop = int(res["status_time"][p]) if failed else last
        templates = [None] * O

        def make_templates(t, ps, w):
            for o in np.nonzero(mask[p] & (template_frame == t))[0]:
                img = int(image_index[t, o])
                cam = observers[o].cams[img]
                uv0 = orc.project(cam, orc.weighted_mean(ps, w)[None, 0:3]).ravel()
                box = orc.snap_tile_box(uv0, tile_size, cam[6:8].astype(int))
                tile, cdf = orc.prepare_tile(observers[o].frames[img][box[1]:box[3], box[0]:box[2]], size=highpass_size,
                                             exact_median=True)
                templates[o] = {"tile": tile, "cdf": cdf, "duv": uv0 - box.reshape(2, -1).mean(axis=0)}

        tag = f"point {p} time {first}"
        origin = moment_origin(model)
        ps0 = orc.init_particles(model, init_draws(init[p], model.tangent))
        if failed and stop == first:
            try:
                make_templates(first, ps0, np.ones(len(ps0)))
            except (IndexError, ValueError):
                rep.count("failed points")
                continue
            raise AssertionError(f"{tag}: the device failed (status {res['status'][p]}), the replay does not")
        got = res["particles"][p, first]
        assert (np.abs(got - ps0) <= PROP_TOL * (1 + np.abs(ps0))).all(), f"{tag}: initial particles"
        assert (res["weights"][p, first] == 1.0).all(), f"{tag}: initial weights"
        make_templates(first, got, res["weights"][p, first])
        check_moments(rep, res, p, first, cov, tag, origin)
        for t in range(first + 1, stop + 1):
            tag = f"point {p} time {t}"
            k = t - first - 1
            prev, w_prev = res["particles"][p, t - 1], res["weights"][p, t - 1]
            evolved = prev.copy()
            orc.evolve_particles(model, evolved, taus[t - 1], step_draws(step[p, k], model.tangent))
            if failed and t == stop:
                raise AssertionError(f"{tag}: the device failed (status {res['status'][p]}); the replay has no failure here")
            make_templates(t, evolved, w_prev)
            terms, observed = [], False
            for o in range(O):
                img = int(image_index[t, o]) if mask[p, o] else -1
                flag = 1
                if img >= 0:
                    cam, tpl = observers[o].cams[img], templates[o]
                    size = tpl["tile"].shape[::-1]
                    uv = orc.project(cam, evolved[:, 0:3])
                    box = orc.search_window(uv, size, cam[6:8].astype(int), kx=kx, ky=ky)
                    flag = 2 if box is None else 0
                    if box is not None:
                        observed = True
                        if windows is not None:
                            want = np.array((box[2] - box[0], box[3] - box[1]))
                            have = np.asarray(windows[p, t, o])
                            if not np.array_equal(have, want):
                                edges = window_edges(uv, size, kx, ky)
                                near = np.abs(edges - np.round(edges)) <= 1e-9  # (left, top, right, bottom)
                                near_dim = np.array((near[0] or near[2], near[1] or near[3]))  # width: x edges, height: y
                                ok = (np.abs(have - want) <= 1).all() and near_dim[have != want].all()
                                assert ok, f"{tag} observer {o}: window {have.tolist()}, oracle {want.tolist()}"
                                print(f"{tag} observer {o}: window {have.tolist()} against {want.tolist()}, box edges {edges.tolist()}")
                                rep.count("window +-1 at integer edges")
                            rep.count("windows")
                        pixels = observers[o].frames[img][box[1]:box[3], box[0]:box[2]]
                        search, _ = orc.prepare_tile(pixels, histogram=tpl["cdf"], size=highpass_size, exact_median=True)
                        sse = orc.ssd_surface(search, tpl["tile"], exact=True)
                        sampled = orc.spline_sample(uv, sse, orc.surface_box(box, size, tpl["duv"]), exact=True, kx=kx, ky=ky)
                        terms.append(sampled * (1 / (2 * observers[o].sigma ** 2)))
                assert int(res["obs_flags"][p, t, o]) == flag, f"{tag} observer {o}: obs_flags {res['obs_flags'][p, t, o]}, oracle {flag}"
            ll = orc.surface_log_likelihood(model, evolved)
            if observed:
                kind = "observed"
                w_pre = orc.weights_from_log_likelihoods(terms + ([ll] if ll is not None else []))
            elif ll is None:
                kind, w_pre = "carried", w_prev
            elif not ll.any():
                kind, w_pre = "uniform", np.ones(len(evolved))
            else:
                kind, w_pre = "dem", orc.weights_from_log_likelihoods([ll])
            rep.count(f"{kind} updates")
            u = unif[p, k]
            children, w_got = res["particles"][p, t], res["weights"][p, t]
            anc, err = recover_ancestors(children, evolved)
            rep.worst(f"propagation ({kind})", err)
            if method in ("systematic", "stratified"):
                assert (np.diff(anc) >= 0).all(), f"{tag}: ancestors decrease at child {int(np.argmax(np.diff(anc) < 0))}"
            order = np.argsort(anc, kind="stable")  # (the identity where the ancestors are sorted)
            same = anc[order][1:] == anc[order][:-1]
            assert (children[order][1:][same] == children[order][:-1][same]).all(), f"{tag}: children of one parent differ"
            assert (w_got[order][1:][same] == w_got[order][:-1][same]).all(), f"{tag}: weights of one parent's children differ"
            ref_w = w_pre[anc]
            if kind in ("carried", "uniform"):
                bad = np.nonzero(w_got != ref_w)[0]
                assert len(bad) == 0, f"{tag}: {kind} weight of child {bad[:5].tolist()}: {w_got[bad[:5]]} against {ref_w[bad[:5]]}"
                delta = 0.0
            else:
                rel = float(np.max(np.abs(w_got - ref_w) / ref_w))
                tol = DEM_REL if kind == "dem" else WEIGHT_REL
                assert rel <= tol, f"{tag}: {kind} weights {rel} from the reference's"
                rep.worst(f"weight rel ({kind})", rel)
                delta = 2 * tol
            if method == "residual":
                check_residual(rep, anc, w_pre, u, delta, kind, tag)
                flipped = ()
            elif method == "choice":
                flipped = check_near_ties(rep, anc, orc.choice_indices(w_pre, u), w_pre, u, delta, kind, tag, choice=True)
            else:
                idx = orc.stratified_indices(w_pre, u) if method == "stratified" else orc.systematic_indices(w_pre, u)
                pos = (np.arange(len(w_pre)) + np.asarray(u)) * (1 / len(w_pre))
                flipped = check_near_ties(rep, anc, idx, w_pre, pos, delta, kind, tag)
            rep.count(f"near-ties ({kind})", len(flipped))
            rep.worst("children of one parent", np.bincount(anc).max())
            rep.worst(f"children of one parent ({kind})", np.bincount(anc).max())
            # the step-by-step flow sums the moments about particle 0 of the previous resampled particles (k_s4c_gather and
            # k_s5_finalize read state_buffer(t - 1)); the pipelined flow about k_init's moment origin
            check_moments(rep, res, p, t, cov, tag, prev[0] if method in STEP_METHODS else origin)
    return rep


def oracle_result(res, P, T, O):
    """An oracle ``TrackResult`` (run with ``trace=True``) in the layout ``replay_track`` takes, with its window sizes."""
    flags = res.skipped.copy()
    out = {"means": res.means, "sigmas": res.sigmas, "particles": res.particles, "weights": res.weights, "obs_flags": flags,
           "status": np.array([0 if e is None else 1 for e in res.errors], dtype=np.int32)}
    out["status_time"] = np.zeros(P, dtype=np.int32)
    win = np.zeros((P, T, O, 2), dtype=np.int32)
    for s in res.trace:
        for o, rec in s.get("obs", {}).items():
            box = rec["box"]
            win[s["p"], s["t"], o] = (box[2] - box[0], box[3] - box[1])
    return out, win


def summary(name, rep):
    keys = sorted(rep)
    return name + ": " + ", ".join(f"{k} {rep[k]:.3g}" if isinstance(rep[k], float) else f"{k} {rep[k]}" for k in keys)

