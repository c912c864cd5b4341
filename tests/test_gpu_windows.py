"""Search windows of designed shapes through every organisation of k_s2_surface, against the oracle.

Each session tracks a distortion-free nadir scene on a 1280 x 960 frame.  It runs once so that the templates are cut, then
at every later time a cloud of particles is forced in per point: a few particles on the corners of a chosen uv rectangle and
the others inside it.  The rectangle fixes the search window ``Su x Sv`` through ``oracle.search_window`` (every box edge lies
a quarter pixel inside its integer, so device and oracle cannot round differently).  Every intermediate is compared with the
oracle's functions, which the stored fixtures pin bit for bit to the reference, at the tolerances of ``test_step_teacher_forced``.

The organisation of a window (``dump_clocks[10]``: 1 interleaved in shared memory, 2 planar, 3 staged, 0 global) is predicted
on the host from the kernel's byte counts and checked for every window; each session also checks that the organisations,
window sizes and surface sizes its row lists actually occurred, so that a later change to a threshold or a budget cannot turn
a case into a silent no-op.  uint8 windows are run with and without TMA loads (``GB_TMA=0``) and must agree bit for bit."""
import warnings

import numpy as np
import pytest

import helpers
from glimpse_b200 import synthetic
from oracle import tracker_oracle as orc
from test_gpu_track import (MOMENT_REL, SAMPLED_ABS, SEARCH_TOL, SSE_REL_CV2, SSE_REL_EXACT, TILE_TOL, UV_TOL_PX, WEIGHT_REL)

pytestmark = pytest.mark.gpu

W, H = 1280, 960
MPP = 0.2          # metres per pixel of the nadir scene: u = x / 0.2 + W / 2, v = -y / 0.2 + H / 2
EDGE = 0.25        # distance of every unrounded box edge from its integer
N = 256
CAP = 65536        # dumped pixels per window
SMEM, SMEM_LARGE = 110 * 1024, 224 * 1024
ORG_NAMES = {1: "interleaved", 2: "planar", 3: "staged", 0: "global"}
FOOTPRINT = [[0, 0, 1, 0, 0], [0, 1, 1, 1, 0], [1, 1, 0, 1, 1], [0, 1, 1, 1, 0]]
GLOBAL_BUDGET = -16000  # no interleaved organisation, and too little for the planar or staged one: global


# ------------------------------------------------------------------------------------------------------------------------
# k_s2_surface's shared-memory needs (tile.cuh tile_bytes_needed*, glimpse_b200.cu s2_smem_bytes), restated to predict the
# organisation of each window
# ------------------------------------------------------------------------------------------------------------------------
def a16(b):
    return (b + 15) // 16 * 16


def template_bytes(tw, th, nvals):
    return 0 if tw * th > 1024 else a16(nvals * 8) * 2 + a16(th * tw * 8)


def need_interleaved(Su, Sv, tw, th, nbins, nvals):
    Mu, Mv = Su - tw + 1, Sv - th + 1
    herm, packed = Mv * (Mu | 1) * 16, (Sv + 4) * (Su + 4) * 4
    return a16(max(herm, packed)) + a16(nbins * 8) + template_bytes(tw, th, nvals) + a16(Sv * ((Su + 3) // 4 * 4) * 4) + a16(nbins * 4)


def need_planar(Su, Sv, tw, th, nbins, nvals):
    Mu, Mv = Su - tw + 1, Sv - th + 1
    r1 = a16(Sv * ((Su + 3) // 4 * 4) * 4)
    packed, planes = (Sv + 4) * (Su + 4) * 4, 2 * a16(Mv * (Mu | 1) * 4)
    return r1 + a16(max(packed, planes)) + a16(nbins * 8) + template_bytes(tw, th, nvals) + a16(nbins * 4)


def need_staged(Su, Sv, tw, th, nbins, nvals):
    Mu, Mv = Su - tw + 1, Sv - th + 1
    b = a16(Su * Sv * 2) + a16((Sv + 4) * (Su + 4) * 4) + a16(nbins * 8) + template_bytes(tw, th, nvals) + a16(nbins * 4)
    return max(b, 2 * a16(Mv * (Mu | 1) * 4))


def launch_smem(tw, th):
    if tw * th <= 1024:
        return SMEM
    return SMEM if need_interleaved(tw + 40, th + 40, tw, th, 1024, 0) <= SMEM else SMEM_LARGE


def organisation(Su, Sv, tw, th, nbins, nvals, tile_bytes, degrees):
    smem = launch_smem(tw, th)
    budget = min(abs(tile_bytes), smem) if tile_bytes is not None else smem
    gen = any(k not in (1, 3) for k in degrees)
    if (tile_bytes is None or tile_bytes >= 0) and need_interleaved(Su, Sv, tw, th, nbins, nvals) <= budget:
        return 1
    if gen:
        return 0
    if need_planar(Su, Sv, tw, th, nbins, nvals) <= budget:
        return 2
    if need_staged(Su, Sv, tw, th, nbins, nvals) <= budget:
        return 3
    return 0


# ------------------------------------------------------------------------------------------------------------------------
# frames
# ------------------------------------------------------------------------------------------------------------------------
def convert_frames(scene, kind, bands):
    """The scene's uint8 grey frames as ``kind`` with ``bands`` bands (each band the texture rolled a little)."""
    rng = np.random.RandomState(5)
    out = []
    for f in scene.observers[0].frames:
        g = np.stack([np.roll(f, 3 * k, axis=k % 2) for k in range(bands)], axis=2) if bands > 1 else f
        if kind == "u8":
            pass
        elif kind == "u8_levels8":  # eight grey levels: long runs of ties in every window
            g = (g // 32) * 32
        elif kind == "u16":
            g = g.astype(np.uint16) * 200 + rng.randint(0, 200, g.shape).astype(np.uint16)
        elif kind == "u16_plateaus":  # plateaus, and regions saturated at 0 and at 65535
            g = np.clip((g.astype(np.int64) // 8) * 2000 - 20000, 0, 65535).astype(np.uint16)
        elif kind == "i16":  # promoted to float64 on the way to the device
            g = (g.astype(np.int16) - 128) * 97 + rng.randint(-40, 40, g.shape).astype(np.int16)
        elif kind in ("f32", "f64"):
            g = ((g.astype(np.float64) + rng.rand(*g.shape)) / 255.0).astype(np.float32 if kind == "f32" else np.float64)
        elif kind in ("f32_signed", "f64_signed"):  # negative values, plateaus, and zeros of both signs
            v = np.round((g.astype(np.float64) - 128.0) / 24.0) * 0.5
            v[(v == 0) & (rng.rand(*v.shape) < 0.5)] = -0.0
            g = v.astype(np.float32 if kind == "f32_signed" else np.float64)
        else:
            raise ValueError(kind)
        out.append(np.ascontiguousarray(g))
    scene.observers[0].frames = out
    return scene


def make_scene(kind, bands, tile, n_points, n_frames, seed):
    margin = max(tile) // 2 + 40
    scene = synthetic.nadir_scene(seed=seed, n_points=n_points, n_particles=N, n_frames=n_frames, imgsz=(W, H), distortion=False,
                                  tile_size=tile, margin_px=margin)
    raster = kind.endswith("_raster")
    scene = convert_frames(scene, kind.replace("_raster", ""), bands)
    return synthetic.as_raster_frames(scene) if raster else scene


# ------------------------------------------------------------------------------------------------------------------------
# designed clouds
# ------------------------------------------------------------------------------------------------------------------------
def world_of(uv):
    return np.column_stack(((uv[:, 0] - W / 2) * MPP, -(uv[:, 1] - H / 2) * MPP))


def cloud(box, tile, rng):
    """N particles whose search window is ``box`` = (left, top, right, bottom) integers: the unrounded box edges lie EDGE
    inside them.  Needs right - left >= tile + k + 1 along each axis (no widening by search_window)."""
    l, t, r, b = box
    tw, th = tile
    u0, u1 = l + EDGE + tw / 2, r - EDGE - tw / 2
    v0, v1 = t + EDGE + th / 2, b - EDGE - th / 2
    uv = np.column_stack((rng.uniform(u0, u1, N), rng.uniform(v0, v1, N)))
    uv[:4] = [(u0, v0), (u1, v0), (u0, v1), (u1, v1)]
    ps = np.zeros((N, 6))
    ps[:, 0:2] = world_of(uv)
    ps[:, 3:5] = rng.randn(N, 2) * 0.3
    return ps


def place(size, centre):
    """Integer box of ``size`` = (Su, Sv) around ``centre``, inside the frame."""
    Su, Sv = size
    l = int(min(max(round(centre[0] - Su / 2), 0), W - Su))
    t = int(min(max(round(centre[1] - Sv / 2), 0), H - Sv))
    return (l, t, l + Su, t + Sv)


def mu_pairs(lo, hi, tile):
    """Windows whose surfaces take every Mu and every Mv from lo to hi once (Mv running the other way): odd and even."""
    tw, th = tile
    return [(tw + m - 1, th + (lo + hi - m) - 1) for m in range(lo, hi + 1)]


# ------------------------------------------------------------------------------------------------------------------------
# expected values
# ------------------------------------------------------------------------------------------------------------------------
def exact_ssd(search, tmpl):
    """``orc.ssd_surface(exact=True)`` as one accumulation per template pixel: a float64 sum over the float32-rounded tiles,
    rounded once to float32 (one sliding_window_view expression of a 128 x 128 template over a 225 px window needs about 1 GB)."""
    s = search.astype(np.float32).astype(np.float64)
    t = tmpl.astype(np.float32).astype(np.float64)
    h, w = t.shape
    mv, mu = s.shape[0] - h + 1, s.shape[1] - w + 1
    acc = np.zeros((mv, mu))
    for r in range(h):
        for c in range(w):
            d = s[r:r + mv, c:c + mu] - t[r, c]
            acc += d * d
    out = acc.astype(np.float32)
    out *= 1 / (w * h)
    return out


class Worst(dict):
    def upd(self, key, values):
        v = float(np.max(values)) if np.size(values) else 0.0
        assert np.isfinite(v), f"{key}: non-finite difference (missing or NaN output)"
        self[key] = max(self.get(key, 0.0), v)


def run_session(spec, monkeypatch, worst):
    """One session of a sweep row.  spec: kind, bands, tile, windows (list of (Su, Sv), or ("box", l, t, r, b)), and optionally
    highpass, interpolation, tile_bytes, margin, seed.  Returns the (organisation, Su, Sv, Mu, Mv) of every window seen and the
    number of windows out of frame."""
    import torch

    import glimpse_b200 as gb
    from glimpse_b200 import _lib
    from glimpse_b200.session import Session

    tile = tuple(spec["tile"])
    tw, th = tile
    hp = spec.get("highpass", {"size": (5, 5)})
    hp_size, hp_kw = hp.get("size"), {k: v for k, v in hp.items() if k != "size"}
    interp = spec.get("interpolation", {"kx": 3, "ky": 3})
    kx, ky = interp["kx"], interp["ky"]
    windows = spec["windows"]
    steps = spec.get("steps", 2)
    P = -(-len(windows) // steps)
    seed = spec.get("seed", 11)
    scene = make_scene(spec["kind"], spec["bands"], tile, P, steps + 1, seed)
    u8 = scene.observers[0].frames[0].dtype == np.uint8
    float32 = scene.observers[0].frames[0].dtype == np.float32
    observers, models = synthetic.build(scene, gb)
    tracker = gb.Tracker(observers, rng="numpy", highpass=hp, interpolation=interp, window_margin=spec.get("margin", 191))
    datetimes = tracker.datetimes
    index = np.array([[-1 if v is None else int(v) for v in row] for row in tracker.match_datetimes(datetimes)], dtype=np.int32)
    T = len(datetimes)
    taus = np.ones(T - 1)
    rng = np.random.RandomState(seed)
    init = rng.randn(P, N, 6)
    draws = (init, np.zeros((P, T - 1, N, 3)), rng.rand(P, T - 1))
    session = Session(tracker, models, index, taus, tile, np.ones((P, 1), dtype=bool), draws=draws)
    if spec.get("tile_bytes") is not None:
        session.plan.tile_bytes = session.desc.plan.tile_bytes = spec["tile_bytes"]
    dev = session.device
    session.run()
    torch.cuda.synchronize()
    assert (session.buf["status"].cpu().numpy() == 0).all()

    # templates: the oracle's, cut from the oracle's initial particles, against the device's
    obs_spec, specs, _, _ = helpers.oracle_inputs(scene)
    obs_spec = obs_spec[0]
    imgsz = np.array((W, H))
    tmpl = []
    for p in range(P):
        parts = iter((init[p, :, 0:2], init[p, :, 2], init[p, :, 3:6]))
        ps0 = orc.init_particles(specs[p], lambda *shape: next(parts))
        uv0 = orc.project(obs_spec.cams[0], orc.weighted_mean(ps0, np.ones(N))[None, 0:3], obs_spec.correction(0)).ravel()
        box0 = orc.snap_tile_box(uv0, tile, imgsz)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            tile0, cdf0 = orc.prepare_tile(obs_spec.frames[0][box0[1]:box0[3], box0[0]:box0[2]], size=hp_size, **hp_kw)
        mine = session.templates(p)[0]
        np.testing.assert_array_equal(mine["box"], box0)
        worst.upd("template", np.abs(mine["tile"] - tile0))
        vals, qs = mine["histogram"]
        assert len(vals) == len(cdf0[0])
        worst.upd("template", np.abs(vals - cdf0[0]))
        np.testing.assert_array_equal(qs, cdf0[1])
        tmpl.append(dict(tile=tile0, cdf=cdf0, duv=uv0 - box0.reshape(2, -1).mean(axis=0), uv0=uv0))
    assert worst["template"] <= (2e-6 if float32 else TILE_TOL), worst["template"]

    seen, n_out = [], 0
    scale = 1 / (2 * obs_spec.sigma ** 2)
    for s in range(steps):
        t = 1 + s
        evolved = np.zeros((P, N, 6))
        for p in range(P):
            k = p * steps + s
            w_spec = windows[k % len(windows)]
            box = w_spec[1:] if w_spec[0] == "box" else place(w_spec, tmpl[p]["uv0"])
            evolved[p] = cloud(box, tile, rng)
        u = rng.rand(P)
        session.buf["uniforms"][:, t - 1] = torch.as_tensor(u).to(dev)
        f_ev = torch.as_tensor(np.ascontiguousarray(evolved.transpose(0, 2, 1))).to(dev)

        def dumped_step():
            d = {
                "uv": torch.full((P, 1, N, 2), float("nan"), dtype=torch.float64, device=dev),
                "box": torch.full((P, 1, 4), -1, dtype=torch.int32, device=dev),
                "search": torch.zeros((P, 1, CAP), dtype=torch.float32, device=dev),
                "sse": torch.zeros((P, 1, CAP), dtype=torch.float32, device=dev),
                "sampled": torch.zeros((P, 1, N), dtype=torch.float64, device=dev),
                "weights": torch.zeros((P, N), dtype=torch.float64, device=dev),
                "clocks": torch.full((P, 1, 16), -1, dtype=torch.int64, device=dev),
            }
            io = _lib.gb_stage_io()
            io.force_evolved = f_ev.data_ptr()
            io.dump_uv, io.dump_box = d["uv"].data_ptr(), d["box"].data_ptr()
            io.dump_search, io.dump_sse = d["search"].data_ptr(), d["sse"].data_ptr()
            io.dump_sampled, io.dump_weights = d["sampled"].data_ptr(), d["weights"].data_ptr()
            io.dump_clocks = d["clocks"].data_ptr()
            io.dump_cap = CAP
            session.buf["status"].zero_()
            session.step(t, io)
            torch.cuda.synchronize()
            out = {k: v.cpu().numpy() for k, v in d.items()}
            out["status"] = session.buf["status"].cpu().numpy().copy()
            out["obs_flags"] = session.buf["obs_flags"][:, t, 0].cpu().numpy().copy()
            return out

        got = dumped_step()
        if u8:  # TMA loads (interleaved windows) against ordinary loads: the same bits
            monkeypatch.setenv("GB_TMA", "0")
            plain = dumped_step()
            monkeypatch.delenv("GB_TMA")
            for key in ("uv", "box", "search", "sse", "sampled", "weights", "status", "obs_flags"):
                np.testing.assert_array_equal(plain[key], got[key], err_msg=f"GB_TMA=0 changes {key}")
        weights_ref = np.ones((P, N))  # (a refused point keeps these)
        refused = np.zeros(P, dtype=bool)
        for p in range(P):
            ev = evolved[p]
            uv = orc.project(obs_spec.cams[t], ev[:, 0:3], obs_spec.correction(t))
            box = orc.search_window(uv, tile, imgsz, kx=kx, ky=ky)
            terms = []
            if box is None:
                assert got["obs_flags"][p] == _lib.GB_OBS_OUT_OF_FRAME
                n_out += 1
            else:
                assert got["obs_flags"][p] == 0
                Su, Sv = int(box[2] - box[0]), int(box[3] - box[1])
                Mu, Mv = Su - tw + 1, Sv - th + 1
                ranked = not u8
                if ranked and Su * Sv > 65535:  # the rank pipeline's limit: the point is refused
                    assert got["status"][p] == _lib.GB_ST_WINDOW_TOO_LARGE
                    refused[p] = True
                    seen.append(("refused", Su, Sv, Mu, Mv))
                    continue
                assert got["status"][p] == 0
                worst.upd("uv", np.abs(got["uv"][p, 0] - uv))
                np.testing.assert_array_equal(got["box"][p, 0], box)
                # edges kept away from integers: device and oracle cannot round them differently
                lo, hi = uv.min(axis=0) - np.array(tile) / 2, uv.max(axis=0) + np.array(tile) / 2
                assert np.min(np.abs(np.concatenate((lo, hi)) - np.round(np.concatenate((lo, hi))))) > 1e-6
                pixels = obs_spec.frames[t][box[1]:box[3], box[0]:box[2]]
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    search, _ = orc.prepare_tile(pixels, histogram=tmpl[p]["cdf"], size=hp_size, **hp_kw)
                sse_cv2 = orc.ssd_surface(search, tmpl[p]["tile"])
                sse_ex = exact_ssd(search, tmpl[p]["tile"])
                sbox = orc.surface_box(box, tile, tmpl[p]["duv"])
                sampled = orc.spline_sample(uv, sse_cv2, sbox, kx=kx, ky=ky)
                terms.append(sampled * scale)
                mine_s = got["search"][p, 0, :Sv * Su].reshape(Sv, Su)
                worst.upd("search", np.abs(mine_s - search.astype(np.float32)))
                sse = got["sse"][p, 0, :Mv * Mu].reshape(Mv, Mu)
                worst.upd("sse_cv2", np.abs(sse - sse_cv2) / np.maximum(sse_cv2, 1e-3))
                worst.upd("sse_exact", np.abs(sse - sse_ex) / np.maximum(sse_ex, 1e-3))
                worst.upd("sampled", np.abs(got["sampled"][p, 0] - sampled))
                nbins = 255 * spec["bands"] + 1 if u8 else Su * Sv
                org = organisation(Su, Sv, tw, th, nbins, len(tmpl[p]["cdf"][0]), spec.get("tile_bytes"), (kx, ky))
                clk = got["clocks"][p, 0]
                assert (int(clk[7]), int(clk[8])) == (Su, Sv)
                assert int(clk[10]) == org, (Su, Sv, int(clk[10]), org)
                seen.append((org, Su, Sv, Mu, Mv))
            terms.append(orc.surface_log_likelihood(specs[p], ev))
            weights_ref[p] = orc.weights_from_log_likelihoods([x for x in terms if x is not None])
            worst.upd("weights", np.abs(got["weights"][p] - weights_ref[p]) / weights_ref[p])
        # resampling and moments with the oracle's weights forced in: ancestors bit-exact
        f_w = torch.as_tensor(weights_ref).to(dev)
        idx_dev = torch.full((P, N), -1, dtype=torch.int32, device=dev)
        io2 = _lib.gb_stage_io()
        io2.force_evolved, io2.force_weights, io2.dump_indices = f_ev.data_ptr(), f_w.data_ptr(), idx_dev.data_ptr()
        session.buf["status"].zero_()
        session.step(t, io2)
        torch.cuda.synchronize()
        idx = idx_dev.cpu().numpy()
        means, sig = session.buf["means"].cpu().numpy(), session.buf["sig"].cpu().numpy()
        for p in np.nonzero(~refused)[0]:
            want = orc.systematic_indices(weights_ref[p], u[p])
            np.testing.assert_array_equal(idx[p], want)
            ps, w = evolved[p][want], weights_ref[p][want]
            m_ref = orc.weighted_mean(ps, w)
            s_ref = orc.weighted_sigma(ps, w, m_ref)
            worst.upd("mean", np.abs(means[p, t] - m_ref) / np.maximum(np.abs(m_ref), 1e-3))
            ok = s_ref > 0
            worst.upd("sigma", np.abs(sig[p, t][ok] - s_ref[ok]) / s_ref[ok])
    return seen, n_out, float32, tw * th


def check(worst, float32, area, sse_exact_rel=SSE_REL_EXACT):
    assert worst.get("uv", 0.0) <= UV_TOL_PX
    assert worst.get("search", 0.0) <= (2e-6 if float32 else SEARCH_TOL)
    assert worst.get("sse_cv2", 0.0) <= SSE_REL_CV2
    assert worst.get("sse_exact", 0.0) <= sse_exact_rel * max(1.0, np.sqrt(area / 225.0))
    assert worst.get("sampled", 0.0) <= SAMPLED_ABS
    assert worst.get("weights", 0.0) <= WEIGHT_REL
    assert worst.get("mean", 0.0) <= MOMENT_REL
    assert worst.get("sigma", 0.0) <= 1e-7


# ------------------------------------------------------------------------------------------------------------------------
# the sweep: row -> sessions, and what the row must have covered
# ------------------------------------------------------------------------------------------------------------------------
def spread(lo, hi, n):
    return [int(round(v)) for v in np.linspace(lo, hi, n)]


def cell(kind, bands, tile=(15, 15), **kw):
    """About 20 windows per organisation: interleaved at the production budget; planar, staged and global with the
    interleaved organisation skipped (negative budget); global with a budget too small for the others."""
    sizes = [(s, s) for s in spread(24, 70, 10)] + [(s, s - 7) for s in spread(30, 66, 10)]
    big = [(s, s) for s in spread(60, 150, 20)]
    return [dict(kind=kind, bands=bands, tile=tile, windows=sizes, **kw),
            dict(kind=kind, bands=bands, tile=tile, windows=big, tile_bytes=-SMEM, **kw),
            dict(kind=kind, bands=bands, tile=tile, windows=sizes[::2], tile_bytes=GLOBAL_BUDGET, **kw)]


ALL_ORGS = {1, 2, 3, 0}


def sweep():
    rows = {}
    # SSD lane split (8 / 16 / 32 lanes by Mu) and the clamped last column pair of an odd Mu; th < 4 takes the other ssd_column
    # branch; degree 1 reaches Mu = 3 and 4 (Mu = 2 needs box edges on integers)
    rows["lanes"] = ([dict(kind="u8", bands=1, tile=t, windows=mu_pairs(5, 40, t), steps=3) for t in ((15, 15), (16, 9), (3, 3))]
                     + [dict(kind="u8", bands=1, tile=t, windows=mu_pairs(3, 40, t), steps=3, interpolation={"kx": 1, "ky": 1})
                        for t in ((15, 15), (3, 3))],
                     dict(mu=set(range(3, 41)), mv=set(range(3, 41))))
    # the organisation switches at the production budget
    switches = [(s, s) for s in range(78, 141)] + [(s, 230 - s) for s in range(80, 151, 5)]
    rows["switches"] = ([dict(kind="u8", bands=1, tile=t, windows=switches, steps=4) for t in ((15, 15), (31, 31))],
                        dict(orgs=ALL_ORGS, square=set(range(78, 141))))
    # a 128 x 128 template: the 224 KB launch
    rows["large_224k"] = ([dict(kind="u8", bands=1, tile=(128, 128), windows=[(s, s) for s in range(150, 226, 5)], margin=100)],
                          dict(orgs={1, 3, 0}))
    for kind, bands in (("u8", 1), ("u8", 3), ("u8", 4), ("u8", 5), ("u8", 8), ("u16", 1), ("u16", 3), ("i16", 1),
                        ("f32_raster", 1), ("f64", 1)):
        rows[f"type_{kind}_{bands}"] = (cell(kind, bands), dict(orgs=ALL_ORGS))
    # (the signed float frames with plateaus measured 2.2e-6 from the exact SSD on a B200: float32 rounding of a sum of 225
    # squares, whose bound is 225 * 2^-24 = 1.3e-5; 3e-6 there instead of 2e-6)
    for kind in ("u8_levels8", "u16_plateaus", "f32_signed", "f64_signed"):
        rows[f"ties_{kind}"] = (cell(kind, 1), dict(orgs=ALL_ORGS, sse_exact_rel=3e-6 if "signed" in kind else SSE_REL_EXACT))
    for name, hp in (("size3", {"size": 3}), ("size3x7", {"size": (3, 7)}), ("size4", {"size": 4}),
                     ("const_in", {"size": (3, 5), "mode": "constant", "cval": 0.1, "origin": (1, -2)}),
                     # below every grey level's z-score (about -3.2 here) and above every one (+3.2): the constant sorts first / last
                     ("const_below", {"size": 5, "mode": "constant", "cval": -5.0}),
                     ("const_above", {"size": (5, 3), "mode": "constant", "cval": 5.0}),
                     ("mirror", {"size": 5, "mode": "mirror"}), ("wrap", {"size": (4, 6), "mode": "wrap", "origin": (-2, 2)}),
                     ("nearest", {"size": 7, "mode": "nearest", "origin": 3}),
                     ("footprint", {"footprint": FOOTPRINT, "mode": "mirror", "origin": (0, 1)})):
        rows[f"median_{name}"] = (cell("u8", 1, highpass=hp), dict(orgs=ALL_ORGS))
    for kx, ky in ((2, 2), (4, 5), (5, 2)):  # their only organisations: interleaved and global
        rows[f"degrees_{kx}{ky}"] = (cell("u8", 1, interpolation={"kx": kx, "ky": ky})[::2], dict(orgs={1, 0}))
    for kx, ky in ((1, 3), (3, 1)):
        rows[f"degrees_{kx}{ky}"] = (cell("u8", 1, interpolation={"kx": kx, "ky": ky}), dict(orgs=ALL_ORGS))
    # frame edges: boxes on l = 0, t = 0, r = W, b = H (and corners), then one pixel beyond each
    S = 40
    inside = [("box", 0, 300, S, 300 + S), ("box", 300, 0, 300 + S, S), ("box", W - S, 300, W, 300 + S), ("box", 300, H - S, 300 + S, H),
              ("box", 0, 0, S, S), ("box", W - S, H - S, W, H)]
    beyond = [("box", -1, 300, S - 1, 300 + S), ("box", 300, -1, 300 + S, S - 1), ("box", W - S + 1, 300, W + 1, 300 + S),
              ("box", 300, H - S + 1, 300 + S, H + 1)]
    rows["edges"] = ([dict(kind="u8", bands=1, tile=(15, 15), windows=inside + beyond, steps=2)], dict(out=len(beyond) * 1))
    # the rank pipeline's limit: 255 x 257 = 65 535 pixels is worked on, 256 x 256 refused
    rows["rank_limit"] = ([dict(kind="u16", bands=1, tile=(15, 15), windows=[(255, 257), (257, 255), (256, 256), (60, 60)],
                                steps=1, margin=245)], dict(sizes={(255, 257), (257, 255)}, refused={(256, 256)}))
    # the largest surface a plan allows: Mu = 1024 (window_margin 1023)
    rows["surface_limit"] = ([dict(kind="u8", bands=1, tile=(15, 15), windows=[(15 + 1023, 20), (15 + 1023, 19), (15 + 1000, 22)],
                                   steps=1, margin=1023)], dict(mu={1024}))
    return rows


ROWS = sweep()


@pytest.mark.parametrize("row", list(ROWS))
def test_windows_match_oracle(cuda, monkeypatch, row):
    sessions, want = ROWS[row]
    worst = Worst()
    seen, n_out = [], 0
    float32, area = False, 0
    for k, spec in enumerate(sessions):
        s, o, f32, a = run_session(dict(spec, seed=100 + k), monkeypatch, worst)
        seen += s
        n_out += o
        float32, area = float32 or f32, max(area, a)
    orgs = {e[0] for e in seen if e[0] != "refused"}
    print(row, "windows", len(seen), "organisations", sorted(ORG_NAMES[o] for o in orgs), {k: float(v) for k, v in worst.items()})
    check(worst, float32, area, want.get("sse_exact_rel", SSE_REL_EXACT))
    # planned coverage
    if "orgs" in want:
        assert want["orgs"] <= orgs, (want["orgs"], orgs)
    if "mu" in want:
        assert want["mu"] <= {e[3] for e in seen}
    if "mv" in want:
        assert want["mv"] <= {e[4] for e in seen}
    if "square" in want:
        assert want["square"] <= {e[1] for e in seen if e[1] == e[2]}
    if "sizes" in want:
        assert want["sizes"] <= {(e[1], e[2]) for e in seen if e[0] != "refused"}
    if "refused" in want:
        assert want["refused"] <= {(e[1], e[2]) for e in seen if e[0] == "refused"}
    if "out" in want:
        assert n_out == want["out"]


def test_sweep_plans_its_coverage_on_the_host():
    """The windows each row designs reach the organisations it lists (predicted with the restated byte counts; each GPU session
    then checks the prediction window by window)."""
    for row, (sessions, want) in ROWS.items():
        orgs = set()
        for spec in sessions:
            tw, th = spec["tile"]
            interp = spec.get("interpolation", {"kx": 3, "ky": 3})
            for w in spec["windows"]:
                if w[0] == "box":
                    continue
                Su, Sv = w
                u8 = spec["kind"].startswith("u8")
                if not u8 and Su * Sv > 65535:
                    continue
                nbins = 255 * spec["bands"] + 1 if u8 else Su * Sv
                for nvals in (tw * th // 2, tw * th):
                    orgs.add(organisation(Su, Sv, tw, th, nbins, nvals, spec.get("tile_bytes"), (interp["kx"], interp["ky"])))
        if "orgs" in want:
            assert want["orgs"] <= orgs, (row, want["orgs"], orgs)


@pytest.mark.parametrize("bands", [5, 8])
def test_free_running_uint8_with_5_and_8_bands_matches_oracle(cuda, bands):
    """Tracker.track(rng='numpy') on uint8 frames of 5 and 8 bands (255 * bands + 1 grey levels) against the oracle fed the
    same draws: identical ancestors, moments to 1e-5 sigma."""
    import glimpse_b200 as gb

    scene = synthetic.nadir_scene(seed=41 + bands, n_points=4, n_particles=300, n_frames=5, imgsz=(400, 300), margin_px=100)
    scene = convert_frames(scene, "u8", bands)
    assert scene.observers[0].frames[0].shape == (300, 400, bands)
    observers, models = synthetic.build(scene, gb)
    np.random.seed(4100 + bands)
    tracks = gb.Tracker(observers, rng="numpy").track(models, tile_size=scene.tile_size, return_particles=True)
    assert all(e is None for e in tracks.errors)
    obs, specs, taus, index = helpers.oracle_inputs(scene)
    np.random.seed(4100 + bands)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref = orc.track(obs, specs, taus, index, tile_size=scene.tile_size, return_particles=True)
    same = np.isclose(tracks.particles, ref.particles, rtol=0, atol=1e-9).all(axis=3)
    d = np.abs(tracks.means - ref.means) / np.maximum(ref.sigmas, 1e-12)
    ok = ref.sigmas > 0
    print(bands, "bands: particle mismatch fraction", 1.0 - same.mean(), "max |dmean|/sigma", np.nanmax(d[..., [0, 1, 3, 4]]))
    assert 1.0 - same.mean() <= 1e-4
    assert np.nanmax(d[..., [0, 1, 3, 4]]) <= 1e-5
    assert np.nanmax(np.abs(tracks.sigmas[ok] - ref.sigmas[ok]) / ref.sigmas[ok]) <= 1e-5
