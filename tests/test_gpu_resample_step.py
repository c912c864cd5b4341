"""The step-by-step resamplers (``resample_method='choice'``: k_s4c_scan -> k_s4c_gather; ``'residual'``: k_s4r_residual ->
k_s4c_gather; then k_s5_finalize) teacher-forced at production block counts: one ``gb_track_step`` with forced evolved
particles, forced weights and supplied uniform rows, against the reference's NumPy statements (``oracle.residual_indices``,
``oracle.choice_indices``) fed the same weights and the same row.

N runs from 1 to 1 000 001 particles (1 to 1 303 blocks, ragged last blocks, N = 49, 765 and 99 005 where N (1 / N) rounds
below 1 so that uniform weights give the residual resampler no repetitions and every child is searched).  Every point of a
call carries its own weight design and uniform row (one row draws its keys from the reference's own cumulative sums, so that
one ulp of difference in a device sum moves an ancestor); the call has three observers (three slots per point in the scratch
layout), a point whose status is already non-zero between active points, and its points in batches that start at p0 > 0 and
run on four side streams.

* residual: the ancestors are bit-equal to the reference's (DESIGN §5: restated operation by operation);
* choice: bit-equal where every cumulative weight is exact (ones at power-of-two N, integer weights with a power-of-two
  total, a collapse onto one parent); elsewhere a differing ancestor must be a near-tie within the bound of two summation
  orders of a positive sum, (N + 2) eps C;
* the gathered particles and weights are the forced ones of the ancestors, bit for bit;
* the moments match a long-double reference of the gathered set (``replay.check_moments``)."""
import warnings

import numpy as np
import pytest

import philox
import replay
from glimpse_b200 import synthetic
from oracle import tracker_oracle as orc

pytestmark = pytest.mark.gpu

EPS = np.finfo(float).eps
SIZES = [1, 2, 49, 765, 767, 768, 769, 1537, 9999, 10000, 99005, 131072, 1000001]
ROWS = ["philox", "ascending", "descending", "constant", "alternating", "ties"]
SKIPPED = 1  # the point whose status is non-zero before the step


def weight_designs(N, method, s_block, rng):
    """{name: weights} of one call: uniform, exact sums, collapses (first block, last block, on a block boundary), rand^6,
    DEM-like log-likelihoods over 0..800 (subnormal exp and the 1e-300 floor), and for the residual resampler negative
    residuals and K = N - 1 repetitions."""
    out = {"ones": np.ones(N)}
    r = rng.randint(1, 8, N).astype(float)  # integers with a power-of-two total: every cumulative sum exact in any order
    q, rem = divmod(2.0 ** np.ceil(np.log2(r.sum())) - r.sum(), N)
    r += q
    r[:int(rem)] += 1
    out["pow2_total"] = r
    heavy = {"first": min(N, s_block) // 3, "boundary": s_block - 1, "boundary+1": s_block, "last": N - 1}
    for label, k in heavy.items():
        if k < N and k not in [heavy[x] for x in heavy if f"collapse_{x}" in out]:
            w = np.full(N, 1e-300)
            w[k] = 1.0
            out[f"collapse_{label}"] = w
    out["rand6"] = rng.rand(N) ** 6
    out["ll800"] = orc.weights_from_log_likelihoods([800 * rng.rand(N)])
    if method == "residual":
        out["negative_residuals"] = 3 * rng.rand(N)  # N wn in [0, 2): about half the parents have one repetition
        if N > 1:
            w = np.ones(N)
            w[N // 2] = 1e-300  # N wn = N / (N - 1) >= 1 for all others: K = N - 1
            out["k_n_minus_1"] = w
        out["counts"] = np.maximum(rng.multinomial(N, np.ones(N) / N).astype(float), 1e-300)  # N wn integers: K = N if exact
    return out


def uniform_row(kind, N, p, rng, w, method):
    """A row of uniforms; ``ties``: keys drawn from the reference's own cumulative sums (residual: of the residuals; choice: the
    normalised cdf), so that one ulp of difference in a device sum moves an ancestor."""
    if kind == "ties":
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            wn = w / w.sum()
            if method == "residual":
                r = wn - (N * wn).astype(int)
                cs = np.cumsum(r * (1 / r.sum()))
                cs[-1] = 1.0
            else:
                cs = np.cumsum(wn)
                cs /= cs[-1]
        keys = cs[rng.randint(0, N, N)]
        # (a uniform of 53 bits is 0 or at least 2^-53: a collapse's cumulative weights of k 1e-300 are no positions)
        return np.where((keys >= 2.0 ** -53) & (keys < 1), keys, rng.rand(N))
    if kind == "philox":
        return philox.uniform_particle(replay.SEED, p, 1, np.arange(N, dtype=np.uint64))
    if kind == "ascending":
        return np.sort(rng.rand(N))
    if kind == "descending":
        return np.sort(rng.rand(N))[::-1].copy()
    if kind == "constant":
        return np.full(N, rng.rand())
    assert kind == "alternating"
    return np.where(np.arange(N) % 2 == 0, 0.0, 1 - 2.0 ** -53)


def exact_cumsum(name, N):
    """Designs whose cumulative weights are exact in any summation order (choice must match bit for bit)."""
    return name == "pow2_total" or name.startswith("collapse") or (name == "ones" and N & (N - 1) == 0)


def check_choice(idx, ref, w, u, name, tag):
    """Bit-equal where the cumulative weights are exact; elsewhere every difference a near-tie: the child's position within
    (N + 2) eps C of the cumulative weight C at the boundary it crossed, the parents crossed weighing no more than that."""
    N = len(w)
    flipped = np.nonzero(idx != ref)[0]
    if exact_cumsum(name, N):
        assert len(flipped) == 0, f"{tag}: children {flipped[:5].tolist()} have {idx[flipped[:5]].tolist()}, reference {ref[flipped[:5]].tolist()}"
        return 0
    if len(flipped):
        C = np.cumsum(w / w.sum())
        C /= C[-1]
        a, b = np.minimum(idx[flipped], ref[flipped]), np.maximum(idx[flipped], ref[flipped])
        band = (N + 2) * EPS * C[b - 1]
        gap, between = np.abs(u[flipped] - C[a]), C[b - 1] - C[a]
        bad = np.nonzero((gap > band) | (between > band))[0]
        assert len(bad) == 0, (f"{tag}: children {flipped[bad[:5]].tolist()} have {idx[flipped[bad[:5]]].tolist()}, reference "
                               f"{ref[flipped[bad[:5]]].tolist()}, |u - C| {gap[bad[:5]].tolist()} (band {band[bad[:5]].tolist()})")
    return len(flipped)


@pytest.mark.parametrize("N", SIZES)
@pytest.mark.parametrize("method", ["choice", "residual"])
def test_resampler_teacher_forced(cuda, monkeypatch, method, N):
    import glimpse_b200 as gb
    from glimpse_b200 import _lib
    from glimpse_b200.session import Session

    torch = cuda
    rng = np.random.RandomState(N)
    scene = synthetic.nadir_scene(seed=68, n_points=1, n_particles=N, n_frames=3, imgsz=(320, 240), margin_px=100)
    first = scene.observers[0]
    for _ in range(2):  # three observers with a frame at every time: three slots per point in the scratch layout
        scene.observers.append(synthetic.ObserverScene([f.copy() for f in first.frames], first.cams.copy(), list(first.datetimes),
                                                       first.sigma))
    observers, models = synthetic.build(scene, gb)
    s_block = replay.stream_block(N)
    designs = weight_designs(N, method, s_block, rng)
    if N <= 10000:  # every design with every row
        layout = [(d, r) for d in designs for r in ROWS]
    else:  # each design with one row (every row used) and with ties
        layout = [(d, ROWS[i % (len(ROWS) - 1)]) for i, d in enumerate(designs)] + [(d, "ties") for d in designs]
    layout.insert(SKIPPED, None)
    P = len(layout)
    # one point per batch below 10^5 particles (p0 = 0 .. P - 1 on four side streams); above, four batches of several points,
    # so that the one-CTA-per-point residual kernels of all points run at once
    monkeypatch.setenv("GB_STREAM_BATCH", "1" if N < 100000 else str(-(-P // 4)))
    monkeypatch.setenv("GB_STREAM_SLOTS", "4")
    cov = N % 2 == 1
    T, S = 3, 2
    index = np.tile(np.arange(T, dtype=np.int32)[:, None], (1, 3))
    unif = np.zeros((P, S, N))
    weights = np.ones((P, N))
    for p, item in enumerate(layout):
        if item is not None:
            weights[p] = designs[item[0]]
            unif[p, 0] = uniform_row(item[1], N, p, rng, weights[p], method)
    draws = (np.zeros((P, N, 6)), np.zeros((P, S, N, 3)), unif)
    tracker = gb.Tracker(observers, rng="numpy", resample_method=method)
    session = Session(tracker, [models[0]] * P, index, np.ones(T - 1), scene.tile_size, np.ones((P, 3), dtype=bool),
                      return_covariances=cov, return_particles=True, draws=draws)
    assert session.plan.stream_block == s_block and session.plan.n_observers == 3
    ev = np.empty((P, N, 6))
    ev[:, :, 0:2] = scene.points[0] + 5 * rng.randn(P, N, 2)
    ev[:, :, 2] = 100 + rng.randn(P, N)
    ev[:, :, 3:6] = 0.3 * rng.randn(P, N, 3)
    dev = session.device
    f_ev = torch.as_tensor(np.ascontiguousarray(ev.transpose(0, 2, 1))).to(dev)
    f_w = torch.as_tensor(weights).to(dev)
    i_dump = torch.full((P, N), -1, dtype=torch.int32, device=dev)
    io = _lib.gb_stage_io()
    io.force_evolved, io.force_weights, io.dump_indices = f_ev.data_ptr(), f_w.data_ptr(), i_dump.data_ptr()
    session.buf["status"].zero_()
    session.buf["status"][SKIPPED] = 3
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    session.step(1, io)
    stop.record()
    torch.cuda.synchronize()
    ms = start.elapsed_time(stop)
    status = session.buf["status"].cpu().numpy()
    assert status[SKIPPED] == 3 and (np.delete(status, SKIPPED) == 0).all(), status
    idx = i_dump.cpu().numpy().astype(np.int64)
    parts = session.buf["particles"][:, 1].cpu().numpy()
    wts = session.buf["weights"][:, 1].cpu().numpy()
    means = session.buf["means"][:, 1].cpu().numpy()
    sig = session.buf["sig"][:, 1].cpu().numpy()
    assert (idx[SKIPPED] == -1).all() and np.isnan(means[SKIPPED]).all() and np.isnan(wts[SKIPPED]).all()
    res = {"particles": parts[:, None], "weights": wts[:, None], "means": means[:, None],
           "sigmas": sig.reshape(P, 1, 6, 6) if cov else sig[:, None]}
    rep = replay.Report()
    for p, item in enumerate(layout):
        if item is None:
            continue
        name, row = item
        tag = f"{method} N {N} point {p} ({name}, {row} row)"
        w, u = weights[p], unif[p, 0]
        if method == "residual":
            with warnings.catch_warnings():  # N = 1: no residual left, 1 / 0 (NumPy's statements as they are)
                warnings.simplefilter("ignore")
                ref, used = orc.residual_indices(w, lambda m: u[:m])
            K = N - len(used)
            rep.count(f"K = {'N' if K == N else 'N - 1' if K == N - 1 else '0' if K == 0 else 'other'}")
            bad = np.nonzero(idx[p] != ref)[0]
            assert len(bad) == 0, f"{tag}: K {K}, children {bad[:5].tolist()} have {idx[p, bad[:5]].tolist()}, reference {ref[bad[:5]].tolist()}"
        else:
            ref = orc.choice_indices(w, u)
            rep.count("near-ties", check_choice(idx[p], ref, w, u, name, tag))
        assert np.array_equal(parts[p], ev[p][idx[p]]), f"{tag}: gathered particles"
        assert np.array_equal(wts[p], w[idx[p]]), f"{tag}: gathered weights"
        # moments about particle 0 of the forced particles, up to 20 m from a collapsed cloud: one pass over a chain of up to
        # 1 303 block partials
        replay.check_moments(rep, res, p, 0, cov, tag, ev[p, 0], terms=16 + -(-N // s_block))
    print(replay.summary(f"{method} N {N}: {P - 1} points, step {ms:.1f} ms", rep))
    if method == "residual":  # the designs keep every case of K the residual resampler has
        assert rep["K = N"] >= 1 and (N == 1 or rep["K = N - 1"] >= 1)
        if N in (49, 765, 99005):
            assert rep["K = 0"] >= 1
