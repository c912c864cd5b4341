"""``Tracker``: drop-in for the reference particle filter (``track/tracker.py:21-625``).

Same constructor and ``track()`` signature, same returned :class:`Tracks`; the per-point,
per-frame work (motion step, projection, tile pipeline, likelihood, resampling, moments) runs in
the sm_100a kernels behind ``gb_track``.  The host keeps what the reference also does on the host:
datetime matching, observer masks, error / warning materialisation.

Differences a user can see (all documented in DESIGN.md):

* ``rng="philox"`` (default) draws on the device from Philox4x32-10, keyed by ``seed`` (or by one
  ``np.random.randint`` draw, so ``np.random.seed`` still makes runs reproducible).  ``rng="numpy"``
  supplies the reference's exact legacy-MT19937 draw sequence (parity runs; ~2.5e7 normals/s).
* ``mode`` is kept for compatibility and must be ``"stream"`` (kernels over all points, batches of points on their own
  streams); round 1's cluster-per-point kernel was removed.
* A track whose work buffers do not fit the device memory that is free runs as consecutive blocks of points (points are
  independent and the device draws are keyed by the global point index, so the results do not depend on the blocks);
  ``max_points`` caps the block size by hand.
* Search windows: every point owns a surface region for windows up to ``window_margin`` (191) px larger than the template.  A
  point whose particle cloud outgrows it (loss of lock after hundreds of frames) is run again on its own with a capacity of 1000 px —
  the device draws are counter-based, so the second run retraces the first one exactly and carries on where it stopped
  (``rng="numpy"`` cannot replay its draws: such a point keeps its ``MemoryError`` in ``Tracks.errors``).
* ``parallel`` is accepted and ignored: points are spread over the GPU, and over ranks when
  ``torch.distributed`` is initialised (one contiguous block of points per rank, one final gather).
* every ``resample_method`` ('systematic', 'stratified', 'residual', 'choice'), ``highpass`` with ``size`` up to 31 x 31 (the default
  5 x 5 'reflect' has the fast kernel) or a ``footprint``, any border ``mode`` / ``cval`` / ``origin`` of
  ``scipy.ndimage.median_filter``, and
  ``interpolation`` degrees 1 to 5 per axis have kernels (3 and 1: Hermite form; 2, 4, 5: B-spline coefficients); a smoothing
  factor raises ``NotImplementedError`` (no CPU fallback).  'residual' with ``rng="numpy"`` cannot replay the reference's
  draws (their number depends on the weights) and raises too.
"""
from __future__ import annotations

import ctypes as C
import datetime as _dt
import warnings as _warnings
from typing import Any, Callable, Iterable, List, Optional, Union

import numpy as np

from . import _lib
from .tracks import Tracks

OUT_OF_FRAME_MESSAGE = "Particles too close to or beyond image bounds, skipping image"


def pairwise_distance_datetimes(x, y) -> np.ndarray:
    """|x_i - y_j| in seconds (reference helpers.py:1831-1854)."""
    xs = np.array([v.timestamp() for v in x], dtype=float)
    ys = np.array([v.timestamp() for v in y], dtype=float)
    return np.abs(xs[:, None] - ys[None, :])


from .session import check_observer_slots, point_span  # noqa: E402,F401  (point_span: re-exported)


def highpass_params(highpass: dict):
    """``scipy.ndimage.median_filter(tile, **highpass)`` (reference tracker.py:59, 530) as the device kernels take it:
    ``(rows, columns, mode, origin_rows, origin_columns, cval, footprint rows as bit masks or None)``.

    ``size`` (one integer or a pair, 1..31 each) or a ``footprint`` (2-D, up to 31 x 31; it wins over ``size``, as in scipy),
    ``mode`` ('reflect' default, 'constant', 'nearest', 'mirror', 'wrap' and their 'grid-' aliases), ``cval`` and ``origin``
    (one integer or a pair)."""
    extra = set(highpass) - {"size", "footprint", "mode", "origin", "cval"}
    if extra:
        raise TypeError(f"median_filter() got an unexpected keyword argument {sorted(extra)[0]!r}")
    footprint = highpass.get("footprint")
    masks = None
    if footprint is not None:
        footprint = np.asarray(footprint, dtype=bool)
        if footprint.ndim != 2 or not footprint.any():
            raise RuntimeError("footprint must be a non-empty 2-D array")
        rows, cols = footprint.shape
        if not footprint.all():
            masks = [int(sum(1 << b for b in range(cols) if footprint[a, b])) for a in range(rows)]
    elif "size" in highpass:
        size = highpass["size"]
        rows, cols = (size, size) if np.ndim(size) == 0 else tuple(size)
    else:
        raise RuntimeError("no footprint or filter size provided")  # scipy's own complaint
    if int(rows) != rows or int(cols) != cols or not (1 <= rows <= 31 and 1 <= cols <= 31):
        raise NotImplementedError("highpass: the window must have between 1 and 31 rows and columns")
    mode = highpass.get("mode", "reflect")
    if mode not in _lib.GB_HP_MODES:
        raise RuntimeError(f"boundary mode not supported: {mode}")  # scipy's own complaint
    origin = highpass.get("origin", 0)
    org_r, org_c = (origin, origin) if np.ndim(origin) == 0 else tuple(origin)
    for org, m in ((org_r, rows), (org_c, cols)):
        if int(org) != org or not (-(int(m) // 2) <= org <= (int(m) - 1) // 2):
            raise ValueError("invalid origin")  # scipy's own complaint
    return int(rows), int(cols), _lib.GB_HP_MODES[mode], int(org_r), int(org_c), float(highpass.get("cval", 0.0)), masks


def highpass_size(highpass: dict):
    """(rows, columns) of the median high-pass (see :func:`highpass_params`)."""
    return highpass_params(highpass)[:2]


def template_size(tile_size):
    """(w, h) of ``Tracker.track(tile_size=...)``.  Templates up to 1024 pixels take any shape; larger ones have a kernel up to
    128 pixels a side, and beyond that ``NotImplementedError`` is raised (there is no CPU fallback)."""
    tw, th = (int(v) for v in tile_size)
    side = _lib.GB_MAX_TEMPLATE_SIDE
    if tw * th > _lib.GB_MAX_TEMPLATE and (tw > side or th > side):
        raise NotImplementedError(f"tile_size: templates above {_lib.GB_MAX_TEMPLATE} pixels have a device kernel up to {side} x {side} "
                                  f"pixels, not {tw} x {th}")
    return tw, th


def interpolation_degrees(interpolation: dict):
    """(kx, ky) of ``RectBivariateSpline(rows, columns, sse, **interpolation)`` (reference tracker.py:60, 584-594,
    observer.py:210): spline degree along the rows / columns of the SSE surface, 1 to 5 each (3 and 1 keep the Hermite-form
    kernels, the others go through B-spline coefficients).  A smoothing factor or a bounding box has no kernel and raises
    ``NotImplementedError`` (there is no CPU fallback)."""
    kx, ky = interpolation.get("kx", 3), interpolation.get("ky", 3)
    if set(interpolation) - {"kx", "ky", "s"} or interpolation.get("s", 0) != 0:
        raise NotImplementedError("interpolation: only the degrees {'kx', 'ky'} of an interpolating spline (s = 0) have a device kernel")
    if kx not in (1, 2, 3, 4, 5) or ky not in (1, 2, 3, 4, 5):
        raise ValueError("kx, ky must be in [1, 5]")  # FITPACK's own complaint
    return int(kx), int(ky)


def shard_bounds(n_items: int, world_size: int, rank: int):
    """Contiguous block [lo, hi) of ``n_items`` owned by ``rank`` (ceil-sized blocks)."""
    per = -(-n_items // world_size)
    lo = min(rank * per, n_items)
    return lo, min(lo + per, n_items)


class Tracker:
    """Estimate the trajectory of world points through time (reference ``tracker.py:21-70``).

    ``observers`` may be any number of stations (a station that was moved or re-calibrated is a new one), with at most eight
    observers with a frame at the same time: ``track`` raises ``NotImplementedError`` naming the first time index with more,
    before any device work (a time step's cameras are kernel launch parameters)."""

    def __init__(
        self,
        observers: Iterable,
        viewshed=None,
        resample_method: str = "systematic",
        highpass: dict = {"size": (5, 5)},
        interpolation: dict = {"kx": 3, "ky": 3},
        *,
        rng: str = "philox",
        seed: Optional[int] = None,
        mode: str = "stream",
        device=None,
        distributed: bool = True,
        max_points: Optional[int] = None,
        window_margin: int = _lib.GB_WINDOW_MARGIN,
    ) -> None:
        self.observers = list(observers)
        self.viewshed = viewshed
        self.resample_method = resample_method
        self.highpass = highpass
        self.interpolation = interpolation
        self.rng = rng
        self.seed = seed
        if mode != "stream":
            raise ValueError("mode must be 'stream' (the cluster-per-point kernel of round 1 was removed)")
        self.mode = mode
        self.device = device
        self.distributed = distributed
        self.max_points = max_points
        self.window_margin = window_margin
        self.particles = None
        self.weights = None
        self.templates = None
        self.last_run: dict = {}
        self._frame_cache: dict = {}

    # ------------------------------------------------------------------ reference-visible state
    @property
    def particle_mean(self) -> np.ndarray:
        return np.average(self.particles, weights=self.weights, axis=0)

    @property
    def particle_covariance(self) -> np.ndarray:
        return np.cov(self.particles.T, aweights=self.weights, ddof=0)

    @property
    def datetimes(self) -> np.ndarray:
        return np.unique(np.concatenate([obs.datetimes for obs in self.observers]))

    def reset(self) -> None:
        self.particles = None
        self.weights = None
        self.templates = None

    def clear_device_cache(self) -> None:
        """Forget the frames kept on the device (their upload events are recycled)."""
        free = self.__dict__.setdefault("_event_free", [])
        free.extend(entry[5] for entry in self._frame_cache.values())
        self._frame_cache.clear()

    # ------------------------------------------------------------------ host-side time logic
    def parse_datetimes(self, datetimes, maxdt: _dt.timedelta = _dt.timedelta(0)) -> np.ndarray:
        """(reference tracker.py:425-464)."""
        datetimes = np.asarray(datetimes)
        monotonic = (datetimes[1:] >= datetimes[:-1]).all() or (datetimes[1:] <= datetimes[:-1]).all()
        if not monotonic:
            raise ValueError("Datetimes must be monotonic")
        selected = np.concatenate(((True,), datetimes[1:] != datetimes[:-1]))
        if not all(selected):
            _warnings.warn("Dropping duplicate datetimes")
            datetimes = datetimes[selected]
        distances = pairwise_distance_datetimes(datetimes, self.datetimes)
        selected = distances.min(axis=1) <= abs(maxdt.total_seconds())
        if not all(selected):
            _warnings.warn("Dropping datetimes not matching any Observers")
            datetimes = datetimes[selected]
        if len(datetimes) < 2:
            raise ValueError("Fewer than two valid datetimes")
        return datetimes

    def match_datetimes(self, datetimes, maxdt: _dt.timedelta = _dt.timedelta(0)) -> np.ndarray:
        """Grid (T, O) of matching image indices, ``None`` = no match (reference tracker.py:466-492)."""
        matches = np.full((len(datetimes), len(self.observers)), None)
        for i, observer in enumerate(self.observers):
            distances = pairwise_distance_datetimes(datetimes, observer.datetimes)
            nearest = np.argmin(distances, axis=1)
            matches[:, i] = nearest
            too_far = distances[np.arange(distances.shape[0]), nearest] > abs(maxdt.total_seconds())
            matches[too_far, i] = None
        return matches

    # ------------------------------------------------------------------ the public entry point
    def track(
        self,
        motion_models: Iterable,
        datetimes: Iterable[_dt.datetime] = None,
        maxdt: _dt.timedelta = _dt.timedelta(0),
        tile_size: Iterable[int] = (15, 15),
        observer_mask: np.ndarray = None,
        return_covariances: bool = False,
        return_particles: bool = False,
        reduce_particles: Callable[[np.ndarray, np.ndarray], Any] = None,
        parallel: Union[bool, int] = False,
    ) -> Tracks:
        """Track particles through time (reference ``tracker.py:225-417``)."""
        import time as _time

        clock = [_time.perf_counter()]
        host_ms = {}

        def lap(name):
            now = _time.perf_counter()
            host_ms[name] = host_ms.get(name, 0.0) + 1e3 * (now - clock[0])
            clock[0] = now

        self._lap = lap
        if reduce_particles:
            return_particles = True
        params = dict(motion_models=motion_models, datetimes=datetimes, maxdt=maxdt, tile_size=tile_size,
                      observer_mask=observer_mask, return_covariances=return_covariances,
                      return_particles=return_particles, reduce_particles=reduce_particles, parallel=parallel)
        motion_models = list(motion_models)
        time_unit = motion_models[0].time_unit
        for model in motion_models[1:]:
            if model.time_unit != time_unit:
                raise ValueError("Motion models must have equal time units")
        counts = sorted({int(m.n) for m in motion_models})
        if len(counts) > 1:
            # every motion model may carry its own number of particles (tracker.py:328): the device sessions are uniform in
            # N, so the points are tracked group by group (one group per particle count) and put back in their order
            return self._track_by_particle_count(counts, params)
        if self.resample_method not in _lib.GB_RESAMPLE:
            raise ValueError(f"unknown resample_method {self.resample_method!r}")
        highpass_size(self.highpass)  # raises for what has no device kernel
        interpolation_degrees(self.interpolation)
        template_size(tile_size)
        self.reset()
        ntracks = len(motion_models)
        raise_errors = ntracks < 2
        if datetimes is None:
            datetimes = self.datetimes
        else:
            datetimes = self.parse_datetimes(datetimes=datetimes, maxdt=maxdt)
        if observer_mask is None:
            observer_mask = np.ones((ntracks, len(self.observers)), dtype=bool)
        observer_mask = np.asarray(observer_mask, dtype=bool).reshape(ntracks, len(self.observers))
        matching_images = self.match_datetimes(datetimes=datetimes, maxdt=maxdt)
        image_index = np.array([[-1 if v is None else int(v) for v in row] for row in matching_images], dtype=np.int32)
        check_observer_slots(image_index)
        unit = time_unit.total_seconds()
        taus = np.array([dt.total_seconds() / unit for dt in np.diff(datetimes)], dtype=float)

        # points owned by this rank
        lo, hi, world, rank = 0, ntracks, 1, 0
        dist = None
        if self.distributed:
            try:
                import torch.distributed as dist_mod

                if dist_mod.is_available() and dist_mod.is_initialized() and dist_mod.get_world_size() > 1:
                    dist = dist_mod
                    world, rank = dist.get_world_size(), dist.get_rank()
                    lo, hi = shard_bounds(ntracks, world, rank)
            except ImportError:
                pass
        # One Philox key per track() call, whatever the sharding: blocks of points and ranks draw from the same key, indexed
        # by the global point number (``seed=None``: one draw from the legacy generator, so np.random.seed still reproduces a
        # run; rank 0's draw is used on every rank).
        seed = None
        if self.rng == "philox":
            seed = self.seed if self.seed is not None else int(np.random.randint(0, 2 ** 62))
            if dist is not None and self.seed is None:
                import torch

                dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
                box = torch.tensor([seed], dtype=torch.int64, device=dev)
                dist.broadcast(box, src=0)
                seed = int(box.item())
        lap("prepare")
        n_particles = int(motion_models[0].n) if ntracks else 0
        tile = tuple(int(v) for v in tile_size)
        args = (image_index, taus, tile)
        # (frames are shared between the ranks only if every rank has points: an idle rank opens no session)
        per_rank = -(-ntracks // world)
        share = dist if (dist is not None and (world - 1) * per_rank < ntracks) else None
        # (a rank whose points fit one device session gathers on the devices while it fetches; the same collective as _gather's)
        on_device = (dist, per_rank, world, ntracks) if (dist is not None and dist.get_backend() == "nccl") else None
        self._gathered = False
        local = self._track_local(motion_models[lo:hi], *args, observer_mask[lo:hi], return_covariances, return_particles,
                                  point_offset=lo, dist=share, seed=seed, n_particles=n_particles, gather=on_device)
        rerun = (seed, motion_models[lo:hi], *args, observer_mask[lo:hi], return_covariances, return_particles, lo)
        if dist is None:
            local = self._rerun_large_windows(local, *rerun)
        else:
            # points are independent: the only collective of the data path is this gather of the result blocks (one call).
            # Every rank then sees every status, so all ranks agree without another collective on whether some points need
            # their second run (a search window that outgrew the plan's capacity) and a second gather.
            lap("local")
            merged = local if self._gathered else self._gather(dist, local, ntracks, world)
            failed = np.nonzero(merged["status"] == _lib.GB_ST_WINDOW_TOO_LARGE)[0]
            if self._can_rerun(seed) and len(failed):
                # every rank runs its own failed points again and the patched rows alone are gathered (padded to the largest
                # count of any rank, which all ranks know from the gathered statuses)
                merged = {k: (v if v.flags.writeable else np.array(v)) for k, v in merged.items()}
                mine = failed[(failed >= lo) & (failed < hi)] - lo
                rows = self._rerun_rows(mine, *rerun)
                counts = [int(((failed >= r * per_rank) & (failed < (r + 1) * per_rank)).sum()) for r in range(world)]
                most = max(counts)
                if rows is None:  # (a rank without failed points contributes padding of the right shapes)
                    rows = {k: v[:0] for k, v in merged.items()}
                patched = self._gather(dist, rows, world * most, world, per=most)
                for r in range(world):
                    idx = failed[(failed >= r * per_rank) & (failed < (r + 1) * per_rank)]
                    for key in merged:
                        merged[key][idx] = patched[key][r * most:r * most + counts[r]]
            local = merged
            lap("gather")

        # materialise errors / warnings the way the reference reports them (tracker.py:358-368)
        errors: List[Optional[BaseException]] = [None] * ntracks
        all_warnings: List[Optional[tuple]] = [None] * ntracks
        status, status_time, flags = local["status"], local["status_time"], local["obs_flags"]
        for p in np.nonzero(status)[0]:
            cls, msg = _lib.GB_ST_MESSAGES[int(status[p])]
            errors[p] = cls(f"{msg} (track {p}, time index {int(status_time[p])})")
        flagged = flags == _lib.GB_OBS_OUT_OF_FRAME
        if flagged.any():
            # warnings raised before a track failed are kept, later ones never happened in the reference
            limit = np.where(status != 0, status_time, flags.shape[1])
            flagged &= np.arange(flags.shape[1])[None, :, None] < limit[:, None, None]
            for p in np.nonzero(flagged.any(axis=(1, 2)))[0]:
                all_warnings[p] = tuple(UserWarning(OUT_OF_FRAME_MESSAGE) for _ in range(int(flagged[p].sum())))
        if raise_errors and errors and errors[0] is not None:
            raise errors[0]
        kwargs = dict(time_unit=time_unit, datetimes=datetimes, means=local["means"], tracker=self,
                      images=matching_images, params=params, errors=errors, warnings=all_warnings)
        particles, weights = local.get("particles"), local.get("weights")
        reduced = None
        if reduce_particles:
            reduced = [reduce_particles(particles[p], weights[p]) for p in range(ntracks)]
            particles = weights = None
        kwargs["particles"], kwargs["weights"] = particles, weights
        if return_covariances:
            kwargs["covariances"] = local["sigmas"]
        else:
            kwargs["sigmas"] = local["sigmas"]
        tracks = Tracks(**kwargs)
        if reduced is not None:
            tracks.reduced = reduced
        lap("results")
        if isinstance(self.last_run, dict):
            self.last_run["host_ms"] = host_ms  # where the wall time of this call went (host view; the device runs under 'fetch')
        return tracks

    def _track_by_particle_count(self, counts, params) -> Tracks:
        models = list(params["motion_models"])
        ntracks, n_obs = len(models), len(self.observers)
        mask = params["observer_mask"]
        mask = np.ones((ntracks, n_obs), dtype=bool) if mask is None else np.asarray(mask, dtype=bool).reshape(ntracks, n_obs)
        user_seed = base_seed = self.seed
        if self.rng == "philox" and base_seed is None:
            base_seed = int(np.random.randint(0, 2 ** 61))
        parts = []
        try:
            for k, n in enumerate(counts):
                idx = [i for i, m in enumerate(models) if int(m.n) == n]
                if base_seed is not None:
                    self.seed = base_seed + k
                kw = dict(params, motion_models=[models[i] for i in idx], observer_mask=mask[idx])
                try:
                    part = self.track(**kw)
                except Exception as exc:  # a group of one point raises instead of capturing: capture it here
                    if ntracks < 2:
                        raise
                    part = exc
                parts.append((idx, part))
        finally:
            self.seed = user_seed
        first = next(part for _, part in parts if isinstance(part, Tracks))
        T = first.means.shape[1]
        cov = first.covariances is not None
        means = np.full((ntracks, T, 6), np.nan)
        sig = np.full((ntracks, T, 6, 6) if cov else (ntracks, T, 6), np.nan)
        errors, warns = [None] * ntracks, [None] * ntracks
        particles = [None] * ntracks if params["return_particles"] and not params["reduce_particles"] else None
        weights = [None] * ntracks if particles is not None else None
        reduced = [None] * ntracks if params["reduce_particles"] else None
        for idx, part in parts:
            for j, i in enumerate(idx):
                if not isinstance(part, Tracks):
                    errors[i] = part
                    continue
                means[i] = part.means[j]
                sig[i] = (part.covariances if cov else part.sigmas)[j]
                errors[i], warns[i] = part.errors[j], part.warnings[j]
                if particles is not None:
                    particles[i], weights[i] = part.particles[j], part.weights[j]
                if reduced is not None:
                    reduced[i] = part.reduced[j]
        kwargs = dict(time_unit=first.time_unit, datetimes=first.datetimes, means=means, tracker=self, images=first.images, params=params,
                      errors=errors, warnings=warns, particles=particles, weights=weights)
        kwargs["covariances" if cov else "sigmas"] = sig
        tracks = Tracks(**kwargs)
        if reduced is not None:
            tracks.reduced = reduced
        return tracks

    # ------------------------------------------------------------------ device plumbing
    def _track_local(self, models, image_index, taus, tile_size, observer_mask, return_covariances, return_particles,
                     point_offset=0, dist=None, seed=None, n_particles=0, gather=None) -> dict:
        """Run the filter for ``models`` on this process's GPU; returns host arrays for these points.  ``dist`` = the NCCL
        group the frames are shared over (only the first session of a call takes part in the shared upload).  Ranks may
        split their points into different numbers of sessions: no collective depends on it."""
        from .session import Session, empty_result

        if len(models) == 0:
            return empty_result(0, image_index.shape[0], image_index.shape[1], return_covariances, return_particles, N=n_particles)
        block = self._points_per_session(models, image_index, tile_size, return_covariances, return_particles)
        # consecutive blocks of points (normally one); the frames stay on the device between them, every block's buffers are
        # released before the next one is planned
        parts, stats = [], None
        for lo in range(0, len(models), block):
            session = Session(self, models[lo:lo + block], image_index, taus, tile_size, observer_mask[lo:lo + block],
                              return_covariances, return_particles, point_offset=point_offset + lo,
                              dist=dist if lo == 0 else None, seed=seed)
            self._lap("session")
            session.run()
            self._lap("enqueue")
            if gather is not None and block >= len(models):
                parts.append(session.fetch(gather))  # results of all ranks
                self._gathered = True
            else:
                parts.append(session.fetch())
            self._lap("fetch")
            st = session.stats
            if stats is None:
                stats = dict(st, sessions=1) if block < len(models) else st
            else:
                stats["sessions"] += 1
                for k in ("kernel_launches", "h2d_bytes", "d2h_bytes"):
                    stats[k] += st[k]
                for k in ("window_width", "window_height"):
                    stats[k] = np.concatenate((stats[k], st[k]))
            if lo + block >= len(models):
                self.particles, self.weights, self.templates = session.final_state()
            del session
        self.last_run = stats
        if len(parts) == 1:
            return parts[0]
        return {k: np.concatenate([part[k] for part in parts], axis=0) for k in parts[0]}

    def _can_rerun(self, seed) -> bool:
        return self.rng == "philox" and seed is not None and self.window_margin < _lib.GB_WINDOW_MARGIN_MAX

    def _rerun_runs(self, failed, seed, models, image_index, taus, tile_size, observer_mask, return_covariances, return_particles,
                    point_offset):
        """Local points ``failed`` (ascending) tracked again with the largest window capacity: yields (first, last + 1, results)
        per run of consecutive points — a session derives the global point numbers its draws are keyed by from its first point.
        The counter-based device draws make the second run identical to the first up to the time it stopped (``seed`` = the
        Philox key of the first run)."""
        from .session import Session

        failed = [int(p) for p in failed]
        runs, start = [], failed[0]
        for a, b in zip(failed, failed[1:] + [None]):
            if b is None or b != a + 1:
                runs.append((start, a + 1))
                start = b
        for lo, hi in runs:
            session = Session(self, models[lo:hi], image_index, taus, tile_size, observer_mask[lo:hi], return_covariances,
                              return_particles, point_offset=point_offset + lo, window_margin=_lib.GB_WINDOW_MARGIN_MAX, seed=seed)
            session.run()
            part = session.fetch()
            del session
            yield lo, hi, part
        self.__dict__.setdefault("_rerun_points", []).extend(int(point_offset + p) for p in failed)

    def _rerun_rows(self, failed, *args):
        """Results of the local points ``failed`` after their second run, in that order (None if there are none)."""
        if len(failed) == 0:
            return None
        parts = [part for _, _, part in self._rerun_runs(failed, *args)]
        return {k: np.concatenate([part[k] for part in parts], axis=0) for k in parts[0]}

    def _rerun_large_windows(self, out, seed, *args) -> dict:
        """Points of ``out`` that ended with GB_ST_WINDOW_TOO_LARGE (their particle cloud outgrew the plan's surface regions)
        are tracked again and their rows replaced in place."""
        failed = np.nonzero(out["status"] == _lib.GB_ST_WINDOW_TOO_LARGE)[0]
        if len(failed) == 0 or not self._can_rerun(seed):
            return out
        for lo, hi, part in self._rerun_runs(failed, seed, *args):
            for key, rows in out.items():
                rows[lo:hi] = part[key]
        return out

    def _points_per_session(self, models, image_index, tile_size, return_covariances, return_particles) -> int:
        """How many points one device session may hold: all of them if their buffers fit 90 % of the device memory that is
        free (counting what the caching allocator can reuse, less the frames still to be uploaded), else the largest block
        that does."""
        from . import session as _session

        torch = _lib.require_cuda()
        P = len(models)
        cap = P if self.max_points is None else max(1, min(P, int(self.max_points)))
        device = torch.device(self.device) if self.device is not None else torch.device("cuda", torch.cuda.current_device())
        frames = 0
        if not self._frame_cache:
            for o, obs in enumerate(self.observers):
                for i in {int(v) for v in image_index[:, o] if v >= 0}:
                    array = getattr(obs.images[i], "array", None)
                    try:
                        frames += int(array.nbytes) if array is not None else 3 * int(np.prod(obs.images[i].size))
                    except (AttributeError, TypeError):
                        pass  # size unknown before the frame is read: the 10 % margin has to cover it
        mode = _lib.GB_MODE_STREAM
        shape = dict(N=int(models[0].n), T=image_index.shape[0], O=image_index.shape[1], tw=tile_size[0], th=tile_size[1],
                     return_covariances=return_covariances, return_particles=return_particles, window_margin=int(self.window_margin),
                     slots=_session.plan_slots(image_index))
        lib = _lib.load()
        # the common case costs no driver call: a track needing less than a quarter of the device is not measured against
        # the free memory (cudaMemGetInfo takes from a fraction of a millisecond to several)
        total = torch.cuda.get_device_properties(device).total_memory
        if _session.session_bytes(lib, mode, 0, cap, **shape) + frames <= total // 4:
            return cap
        free, _total = torch.cuda.mem_get_info(device)
        free += torch.cuda.memory_reserved(device) - torch.cuda.memory_allocated(device)
        return _session.points_per_session(lib, mode, 0, cap, int(0.9 * max(free - frames, 0)), **shape)

    # ------------------------------------------------------------------ multi-GPU: one final gather
    @staticmethod
    def _gather(dist, local: dict, ntracks: int, world: int, per: int = None) -> dict:
        """All-gather the per-rank result blocks in ONE collective (points are independent: no per-step collective): every
        array is padded to the block size ceil(ntracks / world), the blocks are packed into one byte buffer per rank, and the
        gathered buffers are unpacked on the host.  A rank without points contributes arrays of zero rows."""
        import torch

        from .session import result_layout, unpack_results

        backend = dist.get_backend()
        device = torch.device("cuda", torch.cuda.current_device()) if backend == "nccl" else torch.device("cpu")
        per = -(-ntracks // world) if per is None else per
        T, O = local["obs_flags"].shape[1:3]
        cov, parts = local["sigmas"].ndim == 4, "particles" in local
        layout, nbytes = result_layout(per, T, O, local["particles"].shape[2] if parts else 0, cov, parts)
        packed = np.zeros(nbytes, dtype=np.uint8)
        for key, tail, dtype, at, _ in layout:
            arr = np.ascontiguousarray(local[key], dtype=dtype).reshape(-1).view(np.uint8)
            packed[at:at + arr.size] = arr
        mine = torch.from_numpy(packed).to(device)
        if backend == "nccl":
            everyone = torch.empty(world * nbytes, dtype=torch.uint8, device=device)
            dist.all_gather_into_tensor(everyone, mine)
            everyone = everyone.cpu().numpy().reshape(world, nbytes)
        else:
            blocks = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(blocks, mine)
            everyone = np.stack([blk.cpu().numpy() for blk in blocks])
        return unpack_results(everyone, layout, per, ntracks)
