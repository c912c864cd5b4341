"""The replay of tests/replay.py tested on the host: it accepts tracks of the CPU oracle exactly, rejects each of a set of
small corruptions of such a track, and the scenes of tests/test_gpu_replay.py contain the updates that test claims."""
import copy
import warnings

import numpy as np
import pytest

import philox
import replay
from oracle import tracker_oracle as orc


def span(image_index, mask):
    seen = [(image_index[:, m] >= 0).any(axis=1) for m in mask]
    return (np.array([int(np.argmax(s)) for s in seen]), np.array([len(s) - 1 - int(np.argmax(s[::-1])) for s in seen]))


def host_draws(specs, first, last, method, seed):
    """Draws in the layout of ``philox.device_draws``: from NumPy's generator, or (``seed`` = ('philox', key)) the host
    restatement of the device's generator with float64 Box-Muller normals."""
    P, N = len(specs), specs[0].n
    S = max(int((last - first).max()), 1)
    per_particle = method != "systematic"
    if isinstance(seed, tuple):
        key = seed[1]
        init, step = np.zeros((P, N, 6)), np.zeros((P, S, N, 3))
        unif = np.zeros((P, S, N) if per_particle else (P, S))
        n = np.arange(N, dtype=np.uint64)
        for p in range(P):
            f = int(first[p])
            init[p, :, 0:3] = philox.box_muller64(philox.words(key, p, f, n, 0))
            init[p, :, 3:6] = philox.box_muller64(philox.words(key, p, f, n, 1))
            for k in range(int(last[p] - first[p])):
                step[p, k] = philox.box_muller64(philox.words(key, p, f + 1 + k, n, 2))
                unif[p, k] = philox.uniform_particle(key, p, f + 1 + k, n) if per_particle else philox.uniform(key, p, f + 1 + k)
    else:
        rng = np.random.RandomState(seed)
        init, step = rng.randn(P, N, 6), rng.randn(P, S, N, 3)
        unif = rng.random_sample((P, S, N) if per_particle else (P, S))
    for p, m in enumerate(specs):
        if m.tangent:
            init[p, :, 5] = 0.0
    return init, step, unif


def oracle_track(name, n_particles=None, seed=7, method=None):
    """(replay inputs, oracle result, draws) of a replay case run by the oracle with closed-form kernels (``method``: another
    resampler)."""
    scene, mask, method, cov = replay.case(name, n_particles, method)
    inputs = replay.inputs(scene)
    obs, specs, taus, idx = inputs
    first, last = span(idx, mask)
    draws = host_draws(specs, first, last, method, seed)
    P, T, O, N = len(specs), len(taus) + 1, len(obs), specs[0].n
    res = orc.TrackResult(np.full((P, T, 6), np.nan), np.full((P, T, 6, 6) if cov else (P, T, 6), np.nan), [None] * P,
                          np.zeros((P, T, O), dtype=np.uint8), np.full((P, T, N, 6), np.nan), np.full((P, T, N), np.nan), [])
    for p in range(P):  # one call per point: a point that fails stops drawing, the device's draws of the others do not move
        r = philox.replay(*(d[p:p + 1] for d in draws), steps=last[p:p + 1] - first[p:p + 1], tangent=[specs[p].tangent],
                          method=method)
        try:
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                one = orc.track(obs, specs[p:p + 1], taus, idx, tile_size=scene.tile_size, observer_mask=mask[p:p + 1],
                                return_covariances=cov, return_particles=True, exact=True, randn=r.randn, random=r.random,
                                resample_method=method, trace=True)
        except (IndexError, ValueError) as exc:
            res.errors[p] = exc
            continue
        for key in ("means", "sigmas", "skipped", "particles", "weights"):
            getattr(res, key)[p] = getattr(one, key)[0]
        res.trace += [dict(s, p=p) for s in one.trace]
    out, win = replay.oracle_result(res, P, T, O)
    # The oracle's moments are NumPy's average about 0: after a collapse (sigma_x ~ 1e-4 |x|) its float64 rounding reaches
    # 1e-9 sigma.  The device takes them about particle 0, as here.
    for p in range(P):
        for t in range(T):
            ps, w = out["particles"][p, t], out["weights"][p, t]
            if not np.isnan(w).any():
                d = ps - ps[0]
                m = np.average(d, weights=w, axis=0)
                out["means"][p, t] = ps[0] + m
                out["sigmas"][p, t] = np.cov(d.T, aweights=w, ddof=0) if cov else np.sqrt(np.average((d - m) ** 2, weights=w, axis=0))
    args = dict(draws=draws, scene_inputs=inputs, method=method, mask=mask, tile_size=scene.tile_size, cov=cov, windows=win)
    return out, args, res


@pytest.mark.parametrize("name,n", [("small_37", None), ("small_769", None), ("tan_cyl_stratified_odd", 999),
                                    ("cart_dem_floor", 2000), ("tan_carried_collapse", 10000), ("mixed_three_obs", None)])
def test_replay_accepts_oracle_tracks(name, n):
    out, args, _ = oracle_track(name, n)
    rep = replay.replay_track(out, **args)
    print(replay.summary(name, rep))
    for kind in replay.KINDS:
        assert rep.get(f"near-ties ({kind})", 0) == 0
        assert rep.get(f"propagation ({kind})", 0.0) == 0.0
        assert rep.get(f"weight rel ({kind})", 0.0) == 0.0
    assert rep.get("window +-1 at integer edges", 0) == 0 and rep["windows"] > 0
    if name.startswith("small_") or name == "mixed_three_obs":
        assert rep["failed points"] == 1


@pytest.fixture(scope="module")
def collapse():
    """The tangent case at N = 10 000 (14 blocks of 716): its first update is carried (no image for point 0)."""
    out, args, res = oracle_track("tan_carried_collapse", 10000)
    steps = {(s["p"], s["t"]): s for s in res.trace if "indices" in s}
    return out, args, steps


def mutated(out, **changes):
    new = copy.deepcopy(out)
    for key, fn in changes.items():
        fn(new[key])
    return new


def carried_and_observed(args):
    kinds = replay.update_kinds(args["scene_inputs"][1], args["scene_inputs"][3], args["mask"])
    carried = sorted(t for (p, t), k in kinds.items() if p == 0 and k == "carried")
    observed = sorted(t for (p, t), k in kinds.items() if p == 0 and k == "observed")
    return carried, observed


def test_mutations_are_rejected(collapse):
    out, args, steps = collapse
    carried, observed = carried_and_observed(args)
    t_c, t_o = carried[0], observed[0]
    t_c2 = next(t for t in carried if t > t_o)  # carried after an observed update: uneven weights
    anc = np.asarray(steps[(0, t_c)]["indices"])
    evolved = steps[(0, t_c)]["evolved"]
    N = len(anc)

    def swap_across_blocks(ps):  # children 715 | 716 sit on both sides of the first block boundary (blocks of 716)
        assert anc[715] != anc[716]
        ps[0, t_c, [715, 716]] = ps[0, t_c, [716, 715]]

    # a child moved to the next parent where its position is far from that boundary
    C = np.cumsum(np.ones(N) / N)
    pos = (np.arange(N) + steps[(0, t_c)]["u"]) / N
    movable = [i for i in range(N - 1) if anc[i + 1] == anc[i] + 1 and abs(pos[i] - C[anc[i]]) > 0.1 / N
               and (i == 0 or anc[i - 1] != anc[i])]
    i = movable[len(movable) // 2]

    def move(ps):
        ps[0, t_c, i] = evolved[anc[i] + 1]

    single = np.nonzero(np.bincount(np.asarray(steps[(0, t_c2)]["indices"]), minlength=N) == 1)[0]
    j = int(np.searchsorted(np.asarray(steps[(0, t_c2)]["indices"]), single[len(single) // 2]))
    sig = out["sigmas"][0, t_o]

    def drop_block(m):
        ps, w = out["particles"][0, t_o], out["weights"][0, t_o]
        keep = np.ones(N, dtype=bool)
        keep[716:1432] = False
        m[0, t_o] = orc.weighted_mean(ps[keep], w[keep])

    def ulp(w):
        w[0, t_c2, j] = np.nextafter(w[0, t_c2, j], np.inf)

    def shift(m):
        m[0, t_o, 0] += 1e-8 * sig[0]

    cases = {"swap across a block boundary": (mutated(out, particles=swap_across_blocks), None),
             "child moved to the next parent": (mutated(out, particles=move), None),
             "carried weight + 1 ulp": (mutated(out, weights=ulp), None),
             "mean + 1e-8 sigma": (mutated(out, means=shift), None),
             "one block's moments dropped": (mutated(out, means=drop_block), None)}
    win = args["windows"].copy()
    win[0, t_o, 0, 0] += 1
    cases["window width + 1"] = (out, win)
    for label, (bad, windows) in cases.items():
        kw = dict(args, windows=windows) if windows is not None else args
        with pytest.raises(AssertionError) as info:
            replay.replay_track(bad, **kw)
        print(label, "->", str(info.value).splitlines()[0][:160])


def test_edge_uniforms_of_the_reference():
    """The edge uniforms of test_gpu_replay.test_edge_uniforms: at u = 0 the reference's ancestors are [0, 0, 1, ..., N - 2];
    at u = 1 - 2^-53, j + u rounds onto j + 1 for j >= 1, exactly onto the boundaries of N = 2^k equal weights, which
    np.searchsorted's left side gives to the lower parent: [0, 1, ..., N - 1]."""
    for N in (1024, 131072):
        w = np.ones(N)
        np.testing.assert_array_equal(orc.systematic_indices(w, 0.0), np.r_[0, np.arange(N - 1)])
        np.testing.assert_array_equal(orc.stratified_indices(w, np.zeros(N)), np.r_[0, np.arange(N - 1)])
        u = 1 - 2.0 ** -53
        j = np.arange(1, N, dtype=float)
        assert (j + u == j + 1).all() and 0 + u < 1
        np.testing.assert_array_equal(orc.systematic_indices(w, u), np.arange(N))
        np.testing.assert_array_equal(orc.systematic_indices(w, 0.5), np.arange(N))


def test_scenes_contain_what_the_gpu_test_claims():
    """Per replay case: the updates of every kind, the updates where some point starts (k_s4p's speculative prologue off)
    and where none does (on), odd N, a batch with a failed point, the mixed call's three motion kinds, third observer and
    backward times; and, from oracle runs with the host restatement of the philox draws of the GPU test: DEM-only
    log-likelihoods beyond the 1e-300 floor and in the subnormal range of exp, and a parent with more than three chunks of 768 children (at the observed update of the
    collapse: at an update that carries the weights of the last resampling a parent has at most about sqrt(N) / 2
    children, because each child carries its parent's weight, so the carried updates of this case have one or two)."""
    claims = {"tan_carried_collapse": {"carried", "observed"}, "tan_cyl_stratified_odd": {"carried", "observed"},
              "cart_dem_floor": {"dem", "observed"}, "shape_c2_interleaved": {"uniform", "observed"}, "million": {"carried", "observed"},
              "small_2": {"uniform", "observed"}, "small_37": {"uniform", "observed"}, "small_769": {"uniform", "observed"},
              "mixed_three_obs": {"uniform", "dem", "carried", "observed"}}
    starts_late = set()
    for name in replay.CASES:
        scene, mask, method, cov = replay.case(name)
        _, specs, taus, idx = replay.inputs(scene)
        kinds = replay.update_kinds(specs, idx, mask)
        first, last = span(idx, mask)
        counts = {k: sum(1 for v in kinds.values() if v == k) for k in replay.KINDS}
        times = sorted({t for (_, t) in kinds})
        starting = [t for t in times if (first == t).any()]
        print(name, "N", scene.n_particles, "points", len(specs), "updates", counts, "times with a start", starting,
              "without", [t for t in times if t not in starting], "blocks", -(-scene.n_particles // replay.CHUNK))
        assert {k for k, v in counts.items() if v} == claims[name], (name, counts)
        assert any(t not in starting for t in times)
        if starting:
            starts_late.add(name)
    assert starts_late == {"tan_cyl_stratified_odd", "mixed_three_obs"}
    scene, mask, _, _ = replay.case("mixed_three_obs")
    _, specs, taus, idx = replay.inputs(scene)
    first, last = span(idx, mask)
    assert {m.kind for m in specs} == {"cartesian", "cylindrical", "tangent_cartesian"} and (taus < 0).all()
    assert list(first) == [1, 0, 1, 1, 0]
    # observer 2 (slot 2: k_s4p's generic projection loop) has frames at updates of point 4, which sees every observer
    assert mask[4].all() and any(idx[t, 2] >= 0 for t in range(first[4] + 1, last[4] + 1))
    assert {n for n in replay.CASES if replay.case(n)[0].n_particles % 2} == {"tan_cyl_stratified_odd", "million", "small_37",
                                                                               "small_769"}
    out, args, _ = oracle_track("small_37")
    assert list(out["status"]) == [0, 1, 0]
    out, args, _ = oracle_track("mixed_three_obs")
    assert list(out["status"]) == [0, 1, 0, 0, 0]
    out, args, res = oracle_track("cart_dem_floor", seed=("philox", replay.SEED))
    specs = args["scene_inputs"][1]
    kinds = replay.update_kinds(specs, args["scene_inputs"][3], args["mask"])
    ll = np.concatenate([orc.surface_log_likelihood(specs[s["p"]], s["evolved"]) for s in res.trace
                         if "indices" in s and kinds[(s["p"], s["t"])] == "dem"])
    floor, subnormal = int((ll > 745.2).sum()), int(((ll > 708.4) & (ll <= 745.2)).sum())
    print("cart_dem_floor: DEM-only log-likelihoods", ll.min(), "..", ll.max(), ";", floor, "beyond exp's range (weight 1e-300),",
          subnormal, "with a subnormal exp")
    assert floor > 0 and subnormal > 0
    out, args, res = oracle_track("tan_carried_collapse", seed=("philox", replay.SEED))
    most = {s["t"]: int(np.bincount(np.asarray(s["indices"])).max()) for s in res.trace if "indices" in s}
    print("tan_carried_collapse: most children of one parent per time", most)
    assert max(most.values()) > 3 * replay.CHUNK


@pytest.mark.parametrize("name,n,method", [("tan_carried_collapse", 10000, "choice"), ("mixed_three_obs", None, "choice"),
                                           ("tan_cyl_stratified_odd", 999, "residual"), ("cart_dem_floor", 2000, "residual"),
                                           ("small_99005", 2000, "residual")])
def test_replay_accepts_oracle_step_flow_tracks(name, n, method):
    out, args, _ = oracle_track(name, n, method=method)
    rep = replay.replay_track(out, **args)
    print(replay.summary(f"{name} ({method})", rep))
    for kind in replay.KINDS:
        assert rep.get(f"near-ties ({kind})", 0) == 0
        assert rep.get(f"propagation ({kind})", 0.0) == 0.0
        assert rep.get(f"weight rel ({kind})", 0.0) == 0.0
        assert rep.get(f"residual searches within the noise ({kind})", 0) == 0
        assert rep.get(f"residual repetitions off floor(N wn) ({kind})", 0.0) == 0.0
    if name == "mixed_three_obs":
        assert rep["failed points"] == 1


def step_update(steps, t):
    s = steps[(0, t)]
    return np.asarray(s["indices"]), s["evolved"], s["u"]


def test_step_flow_mutations_are_rejected():
    """Choice on the collapse case (N = 10 000, 14 blocks), residual on the odd tangent case (N = 999)."""
    cases = {}
    out, args, res = oracle_track("tan_carried_collapse", 10000, method="choice")
    steps = {(s["p"], s["t"]): s for s in res.trace if "indices" in s}
    carried, observed = carried_and_observed(args)
    t_c, t_o = carried[0], observed[0]
    anc, evolved, _ = step_update(steps, t_c)
    i = 100
    j = next(j for j in range(len(anc) - 1, 0, -1) if anc[j] != anc[i])

    def swap(a):
        a[0, t_c, [i, j]] = a[0, t_c, [j, i]]

    N = len(anc)
    B = replay.stream_block(N)  # the moment partials of the second block

    def drop_block(m):
        ps, w = out["particles"][0, t_o], out["weights"][0, t_o]
        keep = np.ones(N, dtype=bool)
        keep[B:2 * B] = False
        m[0, t_o] = orc.weighted_mean(ps[keep], w[keep])

    cases["choice: two children given each other's parents"] = (mutated(out, particles=swap, weights=swap), args)
    cases["choice: one block's moments dropped"] = (mutated(out, means=drop_block), args)

    out_r, args_r, res_r = oracle_track("tan_cyl_stratified_odd", 999, method="residual")
    steps_r = {(s["p"], s["t"]): s for s in res_r.trace if "indices" in s}
    carried_r, observed_r = carried_and_observed(args_r)
    carried_r = [t for t in carried_r if t > observed_r[0]]  # carried weights of an observed update: uneven
    anc, evolved, u = step_update(steps_r, carried_r[0])
    K = len(anc) - len(u)
    assert 0 < K < len(anc) - 1
    run_end = next(k for k in range(1, K) if anc[k] != anc[k - 1])  # the first parent's repetitions end here

    w_c = steps_r[(0, carried_r[0])]["weights"]

    def shift(ps):  # the first parent gets one more repetition, the next one fewer
        ps[0, carried_r[0], run_end] = evolved[anc[run_end - 1]]

    def shift_w(ws):
        ws[0, carried_r[0], run_end] = w_c[anc[run_end - 1]]

    cases["residual: initial segment shifted by one child"] = (mutated(out_r, particles=shift, weights=shift_w), args_r)
    # an additional child (at an observed update: the noisy path) moved to the next parent, its key far from that parent's and
    # its neighbours' cumulative residuals
    t_o = observed_r[0]
    anc, evolved, u = step_update(steps_r, t_o)
    N = len(anc)
    K = N - len(u)
    w = steps_r[(0, t_o)]["weights"]
    wn = w / w.sum()
    reps = np.bincount(anc[:K], minlength=N)
    cs = np.cumsum((wn - reps) * (1 / (wn - reps).sum()))
    far = [k for k in range(len(u)) if anc[K + k] + 1 < N
           and np.abs(cs[max(anc[K + k] - 1, 0):anc[K + k] + 2] - u[k]).min() > 1e-3]
    k = far[len(far) // 2]

    def move(ps):
        ps[0, t_o, K + k] = evolved[anc[K + k] + 1]

    def move_w(ws):
        ws[0, t_o, K + k] = w[anc[K + k] + 1]

    cases["residual: an additional child moved to the next parent"] = (mutated(out_r, particles=move, weights=move_w), args_r)
    for label, (bad, kw) in cases.items():
        with pytest.raises(AssertionError) as info:
            replay.replay_track(bad, **kw)
        print(label, "->", str(info.value).splitlines()[0][:160])


def test_step_scenes_contain_what_the_gpu_test_claims():
    """The step-flow cases of tests/test_gpu_replay.py: small_99005's uniform updates leave the residual resampler no
    repetitions (N (1 / N) < 1: every child searched), the choice collapse gives a parent more than three blocks of
    children with the philox draws of the GPU test, and the cases keep the kinds of update of their pipelined versions."""
    for name, method in replay.STEP_CASES:
        scene, mask, m, cov = replay.case(name, method=method)
        assert m == method
        _, specs, taus, idx = replay.inputs(scene)
        kinds = replay.update_kinds(specs, idx, mask)
        counts = {k: sum(1 for v in kinds.values() if v == k) for k in replay.KINDS}
        print(name, method, "N", scene.n_particles, "blocks", -(-scene.n_particles // replay.CHUNK), "updates", counts)
        if name == "small_99005":
            N = scene.n_particles
            assert N * (1 / N) < 1 and counts["uniform"] > 0
            assert len(orc.residual_indices(np.ones(N), np.random.random)[1]) == N  # K = 0
    assert replay.case("million", method="choice")[0].n_particles == 1000001
    out, args, res = oracle_track("tan_carried_collapse", seed=("philox", replay.SEED), method="choice")
    most = {s["t"]: int(np.bincount(np.asarray(s["indices"])).max()) for s in res.trace if "indices" in s}
    print("tan_carried_collapse (choice): most children of one parent per time", most)
    assert max(most.values()) > 3 * replay.CHUNK
