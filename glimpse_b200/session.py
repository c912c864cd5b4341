"""Device session of one ``Tracker.track`` call: uploads frames and models, owns every device
buffer, fills the ``gb_track_desc`` and calls the C ABI.  Also used by the parity tests to drive
single teacher-forced steps (``gb_track_init`` / ``gb_track_step``)."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

from itertools import chain as _chain

from . import _lib
from .camera import lower_camera
from .image import Raster


def _struct_array_to_device(torch, structs, ctype, device):
    arr = (ctype * len(structs))(*structs)
    return torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).to(device)


def point_span(image_index: np.ndarray, observer_mask: np.ndarray):
    """first / last time index with an image from a masked observer, per point (reference
    tracker.py:321-325; argmax semantics: a point with no image at all spans the whole sequence)."""
    has = image_index >= 0  # (T, O)
    observed = (observer_mask.astype(np.int64) @ has.T.astype(np.int64)) > 0  # (P, T)
    first = np.argmax(observed, axis=1)
    last = observed.shape[1] - 1 - np.argmax(observed[:, ::-1], axis=1)
    return first.astype(np.int32), last.astype(np.int32)


def empty_result(P, T, O, return_covariances, return_particles, N=0) -> dict:
    out = {
        "means": np.full((P, T, 6), np.nan),
        "sigmas": np.full((P, T, 6, 6) if return_covariances else (P, T, 6), np.nan),
        "status": np.zeros(P, dtype=np.int32), "status_time": np.zeros(P, dtype=np.int32),
        "obs_flags": np.zeros((P, T, O), dtype=np.uint8),
    }
    if return_particles:
        out["particles"], out["weights"] = np.full((P, T, N, 6), np.nan), np.full((P, T, N), np.nan)
    return out


def device_frame(array: np.ndarray) -> np.ndarray:
    """A frame as it is copied to the device: uint8 (the integer tile pipeline), uint16, float32 or float64 (the rank pipeline)
    with 1-8 bands, C-contiguous.  Other integer types go to float64 (exact) and float16 to float32, as NumPy would promote them
    in ``tile.mean(axis=2)`` / ``normalize`` (reference tracker.py:522-526)."""
    if array.ndim not in (2, 3) or (array.ndim == 3 and not 1 <= array.shape[2] <= 8):
        raise NotImplementedError("device frames must be (rows, columns) or (rows, columns, 1-8 bands) arrays")
    if array.dtype.name not in _lib.GB_PIX:
        if array.dtype.kind in "iub":
            array = array.astype(np.float64)
        elif array.dtype == np.float16:
            array = array.astype(np.float32)
        else:
            raise NotImplementedError(f"frames of type {array.dtype} have no device kernel")
    return array if array.flags.c_contiguous else np.ascontiguousarray(array)


class DeviceFrame:
    """A frame that already lies in device memory (``Image.read_device``: decoded there by nvJPEG), dressed like the host
    arrays the upload code handles: shape / dtype / strides / nbytes of the (rows, columns[, bands]) uint8 pixels."""

    def __init__(self, tensor) -> None:
        self.tensor = tensor.contiguous()
        self.shape = tuple(self.tensor.shape)
        self.ndim = self.tensor.dim()
        self.dtype = np.dtype(np.uint8)
        self.nbytes = int(self.tensor.numel())
        self.strides = tuple(int(s) for s in self.tensor.stride())


def frames_need_ranks(observers, image_index) -> bool:
    """Whether some frame a track will read is not uint8 (the surface regions are then sized for rank histograms)."""
    for o, obs in enumerate(observers):
        for i in {int(v) for v in image_index[:, o] if v >= 0}:
            array = getattr(obs.images[i], "array", None)
            if array is not None and array.dtype != np.uint8:
                return True
    return False


def result_layout(per: int, T: int, O: int, N: int, return_covariances: bool, return_particles: bool):
    """Byte layout of one rank's block of results in the gather of a multi-GPU track: ``per`` points per rank (the last
    rank's block is zero-padded), one 16-byte aligned section per array, keys in sorted order.  Returns
    ([(key, shape after the point axis, dtype, offset, bytes)], total bytes)."""
    tails = {"means": ((T, 6), np.float64), "sigmas": ((T, 6, 6) if return_covariances else (T, 6), np.float64),
             "status": ((), np.int32), "status_time": ((), np.int32), "obs_flags": ((T, O), np.uint8)}
    if return_particles:
        tails["particles"], tails["weights"] = ((T, N, 6), np.float64), ((T, N), np.float64)
    layout, at = [], 0
    for key in sorted(tails):
        tail, dtype = tails[key]
        nbytes = per * int(np.prod(tail, dtype=np.int64)) * np.dtype(dtype).itemsize
        layout.append((key, tail, np.dtype(dtype), at, nbytes))
        at += -(-nbytes // 16) * 16
    return layout, at


def unpack_results(everyone: np.ndarray, layout, per: int, ntracks: int) -> dict:
    """``everyone`` = (world, bytes per rank) gathered blocks -> arrays over all points."""
    world = everyone.shape[0]
    merged = {}
    for key, tail, dtype, at, nbytes in layout:
        block = np.ascontiguousarray(everyone[:, at:at + nbytes]).view(dtype).reshape((world * per,) + tuple(tail))
        merged[key] = block[:ntracks]
    return merged


def reference_order_draws(P, N, steps_per_point, tangent=None, stratified=False):
    """Draws from the legacy global NumPy generator in the reference's order (SURVEY.md §8c): per point
    randn(N,2), randn(N), randn(N,3); then per update randn(N,3) and one random().  Points with a tangent model
    (``tangent[p]``) draw randn(N,2), randn(N), randn(N,2); then per update randn(N,2), randn(N) and one random()
    (motion.py:378-420).  The stratified resampler draws random(N) instead of random() (tracker.py:183): ``unif`` is
    then (P, S, N).  Unused slots are 0."""
    S = int(max(steps_per_point)) if len(steps_per_point) else 0
    init = np.zeros((P, N, 6))
    step = np.zeros((P, max(S, 1), N, 3))
    unif = np.zeros((P, max(S, 1), N) if stratified else (P, max(S, 1)))
    for p in range(P):
        tan = bool(tangent[p]) if tangent is not None else False
        init[p, :, 0:2] = np.random.randn(N, 2)
        init[p, :, 2] = np.random.randn(N)
        if tan:
            init[p, :, 3:5] = np.random.randn(N, 2)
        else:
            init[p, :, 3:6] = np.random.randn(N, 3)
        for s in range(int(steps_per_point[p])):
            if tan:
                step[p, s, :, 0:2] = np.random.randn(N, 2)
                step[p, s, :, 2] = np.random.randn(N)
            else:
                step[p, s] = np.random.randn(N, 3)
            unif[p, s] = np.random.random(N) if stratified else np.random.random()
    return init, step, unif


_REFERENCE_MODELS = {  # class name -> (kind, attribute names of v, v_sigma, a, a_sigma)
    "CartesianMotion": (_lib.GB_MOTION_CARTESIAN, ("vxyz", "vxyz_sigma", "axyz", "axyz_sigma")),
    "CylindricalMotion": (_lib.GB_MOTION_CYLINDRICAL, ("vrthz", "vrthz_sigma", "arthz", "arthz_sigma")),
    "TangentCartesianMotion": (_lib.GB_MOTION_TANGENT_CARTESIAN, ("vxy", "vxy_sigma", "axy", "axy_sigma")),
    "TangentCylindricalMotion": (_lib.GB_MOTION_TANGENT_CYLINDRICAL, ("vrth", "vrth_sigma", "arth", "arth_sigma")),
}


class _Adopted:
    """Reference motion-model object (duck-typed by attributes) presented like this package's models."""

    def __init__(self, model, kind, names):
        self._m, self.kind, self._names = model, kind, names
        self.dem, self.dem_sigma, self.n, self.time_unit = model.dem, model.dem_sigma, model.n, model.time_unit
        self.xy, self.xy_sigma = model.xy, model.xy_sigma
        self.slope_sigma = getattr(model, "slope_sigma", 0.0)

    def _velocity(self):
        def pad(x):
            x = tuple(np.asarray(x, dtype=float).ravel())
            return x + (0.0,) * (3 - len(x))

        return tuple(pad(getattr(self._m, n)) for n in self._names)


def adopt_model(model):
    """Built-in models of this package pass through; the reference's are recognised by class name and
    attributes (SURVEY.md §8b).  Anything else has no device kernel."""
    if hasattr(model, "lower"):
        return model
    name = type(model).__name__
    known = _REFERENCE_MODELS.get(name)
    if known is not None and all(hasattr(model, n) for n in known[1]):
        return _Adopted(model, *known)
    raise NotImplementedError(f"motion model {name} has no device kernel (no CPU fallback)")


MOTION_DTYPE = np.dtype([("kind", "<i4"), ("dem", "<i4"), ("dem_sigma", "<i4"), ("pad_", "<i4"), ("xy", "<f8", 2),
                         ("xy_sigma", "<f8", 2), ("v", "<f8", 3), ("v_sigma", "<f8", 3), ("a", "<f8", 3), ("a_sigma", "<f8", 3),
                         ("slope_sigma", "<f8")])  # field layout of gb_motion (include/glimpse_b200.h)


def lower_grid_camera(frame) -> "_lib.gb_camera":
    """Affine ``gb_camera`` of a raster frame: this package's Raster or any object with the reference Grid's ``xlim`` /
    ``ylim`` / ``size`` (raster.py:30-132)."""
    if not (hasattr(frame, "xlim") and hasattr(frame, "ylim") and hasattr(frame, "size")):
        raise NotImplementedError("observer frames must be Image (with .cam) or Raster (with .xlim, .ylim, .size) objects")
    if not isinstance(frame, Raster):
        size = tuple(int(v) for v in frame.size)
        grid = Raster.__new__(Raster)
        grid.array = np.empty((size[1], size[0], 0))  # only the shape is used
        grid.xlim, grid.ylim = np.asarray(frame.xlim, dtype=float), np.asarray(frame.ylim, dtype=float)
        frame = grid
    return frame.lower_grid_camera()


def lower_models(models, viewshed=None):
    """Motion models (this package's or the reference's, SURVEY.md §8b) -> the tables the kernels read, on the host:
    ``(gb_motion table as a structured array, [(gb_surface, cell values or None)], index of the viewshed surface or -1)``.
    Equal constant surfaces (the numbers the models wrap into 0-D rasters, motion.py:136-141) share one entry."""
    assert MOTION_DTYPE.itemsize == C.sizeof(_lib.gb_motion)
    rasters, table, memo = {}, [], {}

    def index_of(raster):
        hit = memo.get(id(raster))
        if hit is not None:
            return hit
        key = getattr(raster, "_const_key", None)
        if key is None or key not in rasters:
            if not (hasattr(raster, "array") and hasattr(raster, "xlim")):
                raise NotImplementedError("motion-model surfaces must be numbers or Raster objects")
            arr = np.asarray(raster.array)
            key = id(raster)
            if arr.ndim != 2 or arr.size == 1:  # constant: share by value (the same key glimpse_b200.Raster gives itself)
                key = "const|%r|%r|%r" % (float(arr.flat[0]), tuple(np.asarray(raster.xlim, dtype=float).tolist()),
                                          tuple(np.asarray(raster.ylim, dtype=float).tolist()))
            if key not in rasters:
                wrapped = raster if isinstance(raster, Raster) else Raster(raster.array, x=raster.xlim, y=raster.ylim)
                rasters[key] = len(table)
                table.append(wrapped.lower_host())
        memo[id(raster)] = out = rasters[key]
        return out

    table_m = np.zeros(len(models), dtype=MOTION_DTYPE)
    adopted = [adopt_model(m) for m in models]
    vel = [m._velocity() for m in adopted]
    table_m["kind"] = [m.kind for m in adopted]
    table_m["dem"] = [index_of(m.dem) for m in adopted]
    table_m["dem_sigma"] = [index_of(m.dem_sigma) for m in adopted]
    n = len(adopted)

    def rows(values, width):
        """(n, width) float64 from n sequences of `width` numbers (flattened through one iterator: several times faster than
        np.array on a list of tuples); anything else — scalars to broadcast, ragged input — takes NumPy's general path."""
        try:
            if isinstance(values[0], np.ndarray):  # (iterating arrays element by element is the slow way round)
                raise TypeError
            out = np.fromiter(_chain.from_iterable(values), dtype=float, count=n * width).reshape(n, width)
        except (TypeError, ValueError):
            out = np.array(values, dtype=float)
            out = np.broadcast_to(out[:, None] if out.ndim == 1 else out, (n, width))
        return out

    table_m["xy"] = rows([m.xy for m in adopted], 2)
    table_m["xy_sigma"] = rows([m.xy_sigma for m in adopted], 2)
    for k, name in enumerate(("v", "v_sigma", "a", "a_sigma")):
        table_m[name] = rows([v[k] for v in vel], 3)
    table_m["slope_sigma"] = [float(getattr(m, "slope_sigma", 0.0)) for m in adopted]
    view = index_of(viewshed) if viewshed is not None else -1
    return table_m, table, view


def observer_slots(image_index: np.ndarray) -> int:
    """Most observers with a matched image at one time in a (T, O) grid of image indices (-1 = no match).  A time step's
    cameras are kernel launch parameters, so this count, not the number of observers, is bounded by ``GB_MAX_OBS``."""
    return int((np.asarray(image_index) >= 0).sum(axis=1).max(initial=0))


def check_observer_slots(image_index: np.ndarray) -> None:
    """Raise ``NotImplementedError`` at the first time with more than ``GB_MAX_OBS`` observers with a matched image."""
    active = (np.asarray(image_index) >= 0).sum(axis=1)
    if active.max(initial=0) > _lib.GB_MAX_OBS:
        t = int(np.argmax(active > _lib.GB_MAX_OBS))
        raise NotImplementedError(f"{int(active[t])} observers have an image at time index {t}: the device kernels take at most "
                                  f"{_lib.GB_MAX_OBS} observers with a frame at the same time")


def plan_slots(image_index: np.ndarray) -> int:
    """Observer slots of a launch plan: one per observer in a call of up to ``GB_MAX_OBS`` observers, otherwise one per
    observer with a frame at the same time (at least one)."""
    O = np.shape(image_index)[1]
    return O if O <= _lib.GB_MAX_OBS else max(observer_slots(image_index), 1)


def plan_template_flags(tw: int, th: int) -> int:
    """The plan flag a ``tw`` x ``th`` template needs: templates above 1024 pixels are planned with their own organisation."""
    return _lib.GB_PLAN_LARGE_TEMPLATES if tw * th > _lib.GB_MAX_TEMPLATE else 0


def plan_flags(observers, image_index, tw: int, th: int) -> int:
    """The flags of a track's launch plan: ranked frames when some frame it reads is not uint8, and the flag of its template size."""
    ranked = _lib.GB_PLAN_RANKED_FRAMES if frames_need_ranks(observers, image_index) else 0
    return ranked | plan_template_flags(tw, th)


def session_bytes(lib, observers, image_index, P: int, N: int, T: int, O: int, tw: int, th: int, return_covariances: bool,
                  return_particles: bool, window_margin: int = _lib.GB_WINDOW_MARGIN, slots: Optional[int] = None) -> int:
    """Device memory one :class:`Session` of ``P`` points allocates (the frames excluded): two particle-state buffers,
    the weights, the launch plan's scratch, templates and result blocks.  ``observers`` / ``image_index``: the frames the
    track reads, which decide the plan's flags (:func:`plan_flags`).  ``slots``: the plan's observer slots
    (:func:`plan_slots`; default ``O``), which size the scratch; templates and results are sized by ``O``."""
    plan = _lib.gb_plan()
    flags = plan_flags(observers, image_index, tw, th)
    _lib.check(lib.gb_step_plan_ex(N, tw, th, P, O if slots is None else int(slots), flags, _lib.GB_MODE_STREAM, int(window_margin),
                                   C.byref(plan)))
    per_point = 2 * 48 * N + 8 * N                      # state_a, state_b, weight_state
    per_point += 3 * O * tw * th * 8 + O * 40           # templates
    per_point += T * ((36 if return_covariances else 6) + 6) * 8 + T * O * 9 + 16  # moments, flags, window sizes, status
    if return_particles:
        per_point += T * N * 56
    return int(plan.scratch_bytes) + P * per_point


def points_per_session(lib, observers, image_index, P: int, budget: int, **shape) -> int:
    """Largest number of points (<= P) whose session fits ``budget`` bytes (at least 1): points are independent, so a
    track that does not fit the device runs as consecutive sessions of this many points."""
    if session_bytes(lib, observers, image_index, P, **shape) <= budget:
        return P
    lo, hi = 1, P  # session_bytes grows with the number of points
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if session_bytes(lib, observers, image_index, mid, **shape) <= budget:
            lo = mid
        else:
            hi = mid
    return lo


class Session:
    def __init__(self, tracker, models, image_index, taus, tile_size, observer_mask, return_covariances=False,
                 return_particles=False, point_offset=0, draws=None, dist=None, window_margin=None, seed=None):
        torch = _lib.require_cuda()
        self.torch = torch
        self.lib = _lib.load()
        self.tracker = tracker
        self.dist = dist  # torch.distributed with an NCCL group spanning the GPUs of the box, or None
        self.device = torch.device(tracker.device) if tracker.device is not None else torch.device("cuda", torch.cuda.current_device())
        self.P, self.T, self.O = len(models), image_index.shape[0], image_index.shape[1]
        P, T, O = self.P, self.T, self.O
        N = self.N = int(models[0].n)
        if any(int(m.n) != N for m in models):
            raise ValueError("one device session holds models with the same number of particles (Tracker.track groups them)")
        check_observer_slots(image_index)
        self.tw, self.th = (int(v) for v in tile_size)
        self.return_covariances, self.return_particles = return_covariances, return_particles
        self.image_index = np.ascontiguousarray(image_index, dtype=np.int32)
        self.taus = np.ascontiguousarray(taus, dtype=float)
        observer_mask = np.asarray(observer_mask, dtype=bool).reshape(P, O)
        device = self.device
        self.keep = []
        with torch.cuda.device(device):
            self.stream = torch.cuda.current_stream().cuda_stream
            self.plan = _lib.gb_plan()
            if window_margin is None:
                window_margin = getattr(tracker, "window_margin", _lib.GB_WINDOW_MARGIN)
            flags = plan_flags(tracker.observers, self.image_index, self.tw, self.th)
            _lib.check(self.lib.gb_step_plan_ex(N, self.tw, self.th, P, plan_slots(self.image_index), flags, _lib.GB_MODE_STREAM,
                                                int(window_margin), C.byref(self.plan)))
            self.h2d = 0
            # the first two frames' uploads start right away (the first kernels wait for them); the other big copies are
            # queued after the small tables, which they would otherwise hold up on the copy engine for tens of ms
            images_dev, self.offsets = self._upload_frames()
            self._start_frame_copies(limit=2)
            motion_dev, surf_dev, n_surf, viewshed = self._lower_models(models)
            self.first, self.last = point_span(self.image_index, observer_mask)
            self.tmpl_frame = np.array([int(np.argmax(self.image_index[:, o] >= 0)) if (self.image_index[:, o] >= 0).any() else -1
                                        for o in range(O)])
            tf = self.tmpl_frame[None, :]
            staggered = bool(np.any(observer_mask & (tf > self.first[:, None]) & (tf >= 0) & (tf <= self.last[:, None])))
            f64, i32, u8 = torch.float64, torch.int32, torch.uint8
            dev = dict(device=device)
            self.mask_h = np.ascontiguousarray(observer_mask.astype(np.uint8))
            self.scale_h = np.array([1 / (2 * obs.sigma ** 2) for obs in tracker.observers], dtype=float)
            self.tau2_h = np.array([float(t) ** 2 for t in self.taus], dtype=float)
            b = self.buf = {}
            b["mask"] = torch.as_tensor(self.mask_h).to(device)
            b["first"], b["last"] = torch.as_tensor(self.first).to(device), torch.as_tensor(self.last).to(device)
            b["state_a"] = torch.empty((P, 6, N), dtype=f64, **dev)
            b["state_b"] = torch.empty((P, 6, N), dtype=f64, **dev)
            # (tangent models keep the weights of the last resampling through updates without any likelihood)
            b["weight_state"] = torch.empty((P, N), dtype=f64, **dev) if (staggered or return_particles or self.tangent.any()) else None
            b["scratch"] = torch.empty((self.plan.scratch_bytes // 8,), dtype=f64, **dev) if self.plan.scratch_bytes else None
            # weights the last point's particles carry when the track ends (Tracker.weights): written at that point's last time only
            b["final_weights"] = torch.ones((N,), dtype=f64, **dev)
            ta = self.tw * self.th
            b["tmpl_tile"] = torch.zeros((P, O, ta), dtype=f64, **dev)
            b["tmpl_values"] = torch.zeros((P, O, ta), dtype=f64, **dev)
            b["tmpl_quantiles"] = torch.zeros((P, O, ta), dtype=f64, **dev)
            b["tmpl_nvalues"] = torch.zeros((P, O), dtype=i32, **dev)
            b["tmpl_box"] = torch.zeros((P, O, 4), dtype=i32, **dev)
            b["tmpl_duv"] = torch.zeros((P, O, 2), dtype=f64, **dev)
            nan = float("nan")
            b["means"] = torch.full((P, T, 6), nan, dtype=f64, **dev)
            b["sig"] = torch.full((P, T, 36 if return_covariances else 6), nan, dtype=f64, **dev)
            b["particles"] = torch.full((P, T, N, 6), nan, dtype=f64, **dev) if return_particles else None
            b["weights"] = torch.full((P, T, N), nan, dtype=f64, **dev) if return_particles else None
            b["status"] = torch.zeros((P,), dtype=i32, **dev)
            b["status_time"] = torch.zeros((P,), dtype=i32, **dev)
            b["obs_flags"] = torch.zeros((P, T, O), dtype=u8, **dev)
            b["window"] = torch.zeros((P, T, O, 2), dtype=i32, **dev)

            d = self.desc = _lib.gb_track_desc()
            d.P, d.N, d.T, d.O, d.tile_w, d.tile_h = P, N, T, O, self.tw, self.th
            d.images = images_dev.data_ptr()
            d.images_host = C.addressof(self.images_host)
            d.image_events_host = C.addressof(self.image_events)
            d.image_offset_host = self.offsets.ctypes.data
            d.image_index_host = self.image_index.ctypes.data
            d.obs_scale_host = self.scale_h.ctypes.data
            d.mask, d.first, d.last = b["mask"].data_ptr(), b["first"].data_ptr(), b["last"].data_ptr()
            d.mask_host, d.first_host, d.last_host = self.mask_h.ctypes.data, self.first.ctypes.data, self.last.ctypes.data
            d.tau_host, d.tau2_host = self.taus.ctypes.data, self.tau2_h.ctypes.data
            d.motion, d.surfaces, d.n_surfaces, d.viewshed = motion_dev.data_ptr(), surf_dev.data_ptr(), n_surf, viewshed
            self.keep += [images_dev, motion_dev, surf_dev]
            d.point_offset = int(point_offset)
            d.motion_kinds = self.motion_kinds
            method = getattr(tracker, "resample_method", "systematic")
            stratified = method in ("stratified", "choice", "residual")  # (up to) one uniform per particle and update
            if method == "residual" and draws is None and tracker.rng == "numpy":
                raise NotImplementedError("resample_method='residual' draws a number of uniforms that depends on the weights: the "
                                          "reference's draw sequence cannot be generated ahead of the run; use rng='philox'")
            d.resample_method = _lib.GB_RESAMPLE[method]
            from .tracker import highpass_params, interpolation_degrees

            rows, cols, hp_mode, org_r, org_c, cval, masks = highpass_params(getattr(tracker, "highpass", {"size": (5, 5)}))
            d.highpass_size = 0 if (rows, cols) == (5, 5) else rows | cols << 16
            d.highpass_mode, d.highpass_origin, d.highpass_cval = hp_mode, (org_r & 0xffff) | (org_c & 0xffff) << 16, cval
            if masks is not None:
                self.footprint_h = np.zeros(31, dtype=np.uint32)
                self.footprint_h[:rows] = masks
                d.highpass_footprint_host = self.footprint_h.ctypes.data
            d.interp_rows, d.interp_cols = interpolation_degrees(getattr(tracker, "interpolation", {}))
            if draws is not None or tracker.rng == "numpy":
                d.rng_mode = _lib.GB_RNG_SUPPLIED
                if draws is None:
                    nbytes = P * max(T - 1, 1) * N * (32 if stratified else 24)
                    if nbytes > 8 << 30:
                        raise MemoryError("rng='numpy' would need %.1f GiB of supplied normals; use rng='philox'" % (nbytes / 2 ** 30))
                    draws = reference_order_draws(P, N, self.last - self.first, self.tangent, stratified)
                init, step, unif = draws
                S = T - 1
                step_full = np.zeros((P, S, N, 3))
                unif_full = np.zeros((P, S, N) if stratified else (P, S))
                step_full[:, : step.shape[1]] = step[:, :S]
                unif_full[:, : unif.shape[1]] = unif[:, :S]
                b["init_normals"] = torch.as_tensor(np.ascontiguousarray(init)).to(device)
                b["step_normals"] = torch.as_tensor(step_full).to(device)
                b["uniforms"] = torch.as_tensor(unif_full).to(device)
                d.init_normals, d.step_normals, d.uniforms = (b[k].data_ptr() for k in ("init_normals", "step_normals", "uniforms"))
                self.h2d += (init.size + step_full.size + unif_full.size) * 8
            elif tracker.rng == "philox":
                d.rng_mode = _lib.GB_RNG_PHILOX
                if seed is None:
                    seed = tracker.seed if tracker.seed is not None else int(np.random.randint(0, 2 ** 62))
                self.seed_used = int(seed)
                d.seed = int(seed) % (1 << 64)
            else:
                raise ValueError("rng must be 'philox' or 'numpy'")
            ptr = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
            d.state_a, d.state_b = ptr(b["state_a"]), ptr(b["state_b"])
            d.weight_state, d.scratch = ptr(b["weight_state"]), ptr(b["scratch"])
            d.final_weights = ptr(b["final_weights"])
            d.tmpl_tile, d.tmpl_values, d.tmpl_quantiles = ptr(b["tmpl_tile"]), ptr(b["tmpl_values"]), ptr(b["tmpl_quantiles"])
            d.tmpl_nvalues, d.tmpl_box, d.tmpl_duv = ptr(b["tmpl_nvalues"]), ptr(b["tmpl_box"]), ptr(b["tmpl_duv"])
            d.means = ptr(b["means"])
            if return_covariances:
                d.covariances = ptr(b["sig"])
            else:
                d.sigmas = ptr(b["sig"])
            d.out_particles, d.out_weights = ptr(b["particles"]), ptr(b["weights"])
            d.status, d.status_time = ptr(b["status"]), ptr(b["status_time"])
            d.obs_flags, d.window_stats = ptr(b["obs_flags"]), ptr(b["window"])
            d.plan = self.plan
            self._start_frame_copies()
        self.launches = 0
        self.stats: dict = {}

    def _start_frame_copies(self, limit=None) -> None:
        """Queue the frame uploads (in time order) on the copy stream, each followed by its event; ``limit`` = only
        the first so many (the rest on the next call).

        With an NCCL group every rank holds the same frames on its host, so they cross PCIe once per box instead of once per
        GPU: the frames lie in a few time-ordered groups of the device arena (``_upload_frames``); of every group each rank
        uploads its 1 / world slice into a staging buffer and ONE ``all_gather_into_tensor`` over NVLink fills the group on
        every GPU (one collective per eight frames instead of one broadcast per frame).  The first group is small, so
        tracking starts while the later groups are still in flight."""
        torch, copy_stream = self.torch, self.tracker._copy_stream
        if not self._shared_upload:
            todo = self._pending_copies if limit is None else self._pending_copies[:limit]
            with torch.cuda.stream(copy_stream):
                for dev, arr, event in todo:
                    src = arr.tensor.reshape(-1) if isinstance(arr, DeviceFrame) else torch.from_numpy(arr).view(torch.uint8).reshape(-1)
                    dev.copy_(src, non_blocking=True)
                    event.record(copy_stream)
            for k, event in self._pending_events:
                self.image_events[k] = event.cuda_event
            self._pending_copies = self._pending_copies[len(todo):]
            return
        if limit is not None or not self._pending_copies:
            if not self._pending_copies:  # every frame was already on the device: their events are recorded
                for k, event in self._pending_events:
                    self.image_events[k] = event.cuda_event
            return  # the bulk groups go out once the small tables are queued (second call)
        dist = self.dist
        world, rank = dist.get_world_size(), dist.get_rank()
        arena = self._arena
        flat = {id(arr): torch.from_numpy(arr).view(torch.uint8).reshape(-1) for _, arr, _ in self._pending_copies}
        with torch.cuda.stream(copy_stream):
            for g0, span, members in self._upload_groups:
                chunk = span // world
                lo, hi = g0 + rank * chunk, g0 + (rank + 1) * chunk
                staging = torch.empty(chunk, dtype=torch.uint8, device=self.device)
                staging.record_stream(copy_stream)
                for off, (dev, arr, event) in members:
                    a, b = max(off, lo), min(off + arr.nbytes, hi)
                    if a < b:  # the part of this frame that lies in this rank's slice of the group
                        staging[a - lo:b - lo].copy_(flat[id(arr)][a - off:b - off], non_blocking=True)
                        self.h2d += b - a
                dist.all_gather_into_tensor(arena[g0:g0 + span], staging)
                for _, (dev, arr, event) in members:
                    event.record(copy_stream)
        # (an event has its handle once it is recorded: the table the kernels wait on is filled afterwards)
        for k, event in self._pending_events:
            self.image_events[k] = event.cuda_event
        self._pending_copies = []

    # ---------------------------------------------------------------- uploads
    def _upload_frames(self):
        """Copy every frame ``image_index`` references to the device as it is (``device_frame``: 1-8 bands; reference
        ``Observer.cache_images`` / ``Image.read``, tracker.py:295-299).  Copies go to a side stream in
        time order, each followed by an event that ``gb_track`` waits on before the first kernel that reads
        the frame, so the upload of later frames overlaps the tracking of earlier ones."""
        torch, device, tracker = self.torch, self.device, self.tracker
        structs, offsets, order = [], [0], []
        for o, obs in enumerate(tracker.observers):
            first_use = {}
            for t, v in enumerate(self.image_index[:, o]):
                if v >= 0:
                    first_use.setdefault(int(v), t)
            for i, img in enumerate(obs.images):
                if i in first_use:
                    order.append((first_use[i], len(structs)))
                structs.append((o, i, img, i in first_use))
            offsets.append(len(structs))
        out = [_lib.gb_image() for _ in structs]
        self.image_events = (C.c_void_p * len(structs))()
        self.keep_events = []
        self._pending_copies = []
        self._pending_events = []
        copy_stream = getattr(tracker, "_copy_stream", None)
        if copy_stream is None or copy_stream.device != device:
            copy_stream = tracker._copy_stream = torch.cuda.Stream(device=device)
        compute_stream = torch.cuda.current_stream(device)
        copy_stream.wait_stream(compute_stream)
        fresh, placed = [], []
        order_of = {k: n for n, (_, k) in enumerate(sorted(order))}
        with torch.cuda.stream(copy_stream):
            for _, k in sorted(order):
                o, i, img, _used = structs[k]
                obs = tracker.observers[o]
                use_cache = bool(getattr(obs, "cache", True))
                on_device = getattr(img, "device_array", None) if getattr(img, "array", None) is None else None
                array = on_device if on_device is not None else (img.array if getattr(img, "array", None) is not None else img.read(cache=use_cache))
                key = (o, i, id(array))
                cached = tracker._frame_cache.get(key) if use_cache else None
                if cached is None:
                    arr = DeviceFrame(array) if on_device is not None else device_frame(array)
                    fresh.append((k, key, use_cache, arr))
                    continue
                placed.append((k, cached))
            # frames not on the device yet: one allocation (on the copy stream) carved into 256-byte aligned slices.
            # Shared upload (NCCL group): the frames form a few time-ordered groups, each padded to a multiple of
            # world x 256 bytes so that every rank contributes an equal slice to the group's all-gather.
            # (frames decoded on the device are copied device to device by every rank itself: nothing to share)
            any_on_device = any(isinstance(arr, DeviceFrame) for _, _, _, arr in fresh)
            self._shared_upload = (not any_on_device) and self._agree_on_shared_upload(len(fresh), sum(arr.nbytes for _, _, _, arr in fresh))
            self._upload_groups = []
            if fresh:
                world = self.dist.get_world_size() if self._shared_upload else 1
                n = len(fresh)
                # groups in time order: two frames first (tracking starts as soon as they are there), then eight at a time —
                # small enough that the uploads stay ahead of the tracking, large enough that a track needs ~n / 8 collectives
                bounds = sorted(set([0, min(n, 2)] + list(range(min(n, 2), n, 8)) + [n]))
                offsets_b, total = [], 0
                for lo_g, hi_g in zip(bounds[:-1], bounds[1:]):
                    g0 = total
                    for _, _, _, arr in fresh[lo_g:hi_g]:
                        offsets_b.append(total)
                        total += (arr.nbytes + 255) // 256 * 256
                    if self._shared_upload:
                        total = g0 + -(-(total - g0) // (world * 256)) * (world * 256)
                        self._upload_groups.append([g0, total - g0, []])
                arena = torch.empty(total, dtype=torch.uint8, device=device)
                arena.record_stream(compute_stream)
                self._arena = arena
                free = tracker.__dict__.setdefault("_event_free", [])  # events handed back by clear_device_cache()
                for n_f, ((k, key, use_cache, arr), off) in enumerate(zip(fresh, offsets_b)):
                    dev = arena[off:off + arr.nbytes]  # (bytes: the frame keeps its own pixel type)
                    event = free.pop() if free else torch.cuda.Event()
                    self._pending_copies.append((dev, arr, event))
                    if self._shared_upload:
                        group = max(g for g in range(len(self._upload_groups)) if self._upload_groups[g][0] <= off)
                        self._upload_groups[group][2].append((off, (dev, arr, event)))
                    elif not isinstance(arr, DeviceFrame):
                        self.h2d += arr.nbytes
                    cached = (dev, arr.shape[1], arr.shape[0], arr.strides[0], 1 if arr.ndim == 2 else arr.shape[2], event,
                              _lib.GB_PIX[arr.dtype.name])
                    if use_cache:
                        tracker._frame_cache[key] = cached
                    placed.append((k, cached))
            for k, cached in sorted(placed, key=lambda kc: order_of[kc[0]]):
                o, i, img, _used = structs[k]
                dev, w, h, pitch, nchan, event, pix = cached
                self.keep.append(dev)
                self.keep_events.append(event)
                g = out[k]
                g.pixels = dev.data_ptr()
                g.width, g.height, g.pitch, g.nchan, g.dtype = w, h, pitch, nchan, pix
                g.cam = self._lower_frame_camera(img)
                self._pending_events.append((k, event))
        self.images_host = (_lib.gb_image * len(out))(*out)
        images_dev = torch.frombuffer(bytearray(bytes(self.images_host)), dtype=torch.uint8).to(device)
        self.h2d += images_dev.numel()
        return images_dev, np.asarray(offsets, dtype=np.int32)

    def _agree_on_shared_upload(self, n_frames: int, n_bytes: int) -> bool:
        """Whether this session's frames are uploaded once per box and shared over NVLink.  All ranks must be about to upload
        the same list (a rank whose frames are still cached would not take part): agreed with one ``all_reduce`` the first
        time a Tracker sees an upload of this size, remembered afterwards — ``track()`` is a collective call under
        ``torch.distributed`` (same arguments, same cache state on every rank), so later sessions need no agreement."""
        dist = self.dist
        if dist is None or dist.get_backend() != "nccl" or os.environ.get("GB_SHARED_UPLOAD", "1") == "0":
            return False
        agreed = self.tracker.__dict__.setdefault("_shared_upload_agreed", {})
        key = (int(n_frames), int(n_bytes))
        if key not in agreed:
            torch = self.torch
            sig = torch.tensor([key[0], key[1], -key[0], -key[1]], dtype=torch.int64, device=self.device)
            dist.all_reduce(sig, op=dist.ReduceOp.MIN)  # min and (negated) max in one call
            sig = sig.tolist()
            agreed[key] = bool(sig[0] == -sig[2] and sig[1] == -sig[3])
        return agreed[key] and n_frames > 0

    def _lower_frame_camera(self, img):
        """``gb_camera`` of one frame: the Image's Camera, or the affine grid map of a Raster frame (an Observer of
        orthoimages: anything with ``xlim`` / ``ylim`` / ``size`` and no ``cam``, reference raster.py:423-445)."""
        cam = getattr(img, "cam", None)
        if cam is not None:
            return self._lower_camera_memo(cam)
        return lower_grid_camera(img)

    def _lower_camera_memo(self, cam):
        """``lower_camera`` once per distinct camera (a sequence of frames usually shares one)."""
        memo = self.__dict__.setdefault("_camera_memo", {})
        vec = getattr(cam, "vector", None)
        if vec is None:
            vec = getattr(cam, "_vector", None)  # the reference's Camera keeps its 20-vector here
        if vec is None:
            return lower_camera(cam)
        corr = getattr(cam, "correction", None)
        key = (np.asarray(vec, dtype=float).tobytes(), tuple(int(v) for v in cam.imgsz),
               tuple(sorted(corr.items())) if isinstance(corr, dict) else None)
        hit = memo.get(key)
        if hit is None:
            hit = memo[key] = lower_camera(cam)
        return hit

    def _lower_models(self, models):
        torch, device = self.torch, self.device
        table_m, surfaces, viewshed = lower_models(models, self.tracker.viewshed)
        table = []
        for s, z in surfaces:
            if z is not None:
                tensor = torch.as_tensor(z).to(device)
                s.z = tensor.data_ptr()
                self.keep.append(tensor)
            table.append(s)
        self.tangent = table_m["kind"] >= _lib.GB_MOTION_TANGENT_CARTESIAN
        self.motion_kinds = int(np.bitwise_or.reduce(1 << table_m["kind"].astype(np.int64))) if len(models) else 0
        motion_dev = torch.from_numpy(table_m.view(np.uint8).reshape(-1)).to(device)
        surf_dev = _struct_array_to_device(torch, table, _lib.gb_surface, device)
        self.h2d += motion_dev.numel() + surf_dev.numel()
        return motion_dev, surf_dev, len(table), viewshed

    # ---------------------------------------------------------------- C-ABI calls
    def run(self) -> None:
        """``gb_track``: every time step for every point, asynchronously on the current stream."""
        launches = C.c_int64(0)
        with self.torch.cuda.device(self.device):
            _lib.check(self.lib.gb_track(C.byref(self.desc), self.stream, C.byref(launches)))
        self.launches += int(launches.value)

    def _await_uploads(self) -> None:
        """Per-time entry points do not take the frame events: wait for the whole copy stream once."""
        if not getattr(self, "_uploads_awaited", False):
            self.torch.cuda.current_stream(self.device).wait_stream(self.tracker._copy_stream)
            self._uploads_awaited = True

    def init(self, t: int) -> None:
        self._await_uploads()
        with self.torch.cuda.device(self.device):
            _lib.check(self.lib.gb_track_init(C.byref(self.desc), int(t), self.stream))

    def step(self, t: int, io: Optional[_lib.gb_stage_io] = None) -> None:
        self._await_uploads()
        with self.torch.cuda.device(self.device):
            _lib.check(self.lib.gb_track_step(C.byref(self.desc), int(t), C.byref(io) if io is not None else None, self.stream))

    # ---------------------------------------------------------------- results
    def fetch(self, gather=None) -> dict:
        """Results to host memory: every array is copied into pinned memory on the compute stream without
        blocking, then one synchronisation covers them all.  ``gather`` = (dist, points per rank, world size, points in
        all): this session holds all of this rank's points, so its result blocks are packed into one byte buffer ON THE
        DEVICE (``result_layout``), all-gathered in one NCCL call, and the returned arrays hold every rank's points."""
        torch, b, P, T = self.torch, self.buf, self.P, self.T
        names = ["means", "sig", "status", "status_time", "obs_flags", "window"]
        if self.return_particles:
            names += ["particles", "weights"]
        host = {}
        with torch.cuda.device(self.device):
            if gather is not None:
                dist, per, world, ntracks = gather
                layout, nbytes = result_layout(per, T, self.O, self.N, self.return_covariances, self.return_particles)
                mine = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
                for key, tail, dtype, at, _ in layout:
                    src = b["sig" if key == "sigmas" else key].reshape(-1).view(torch.uint8)
                    mine[at:at + src.numel()].copy_(src)
                everyone = torch.empty(world * nbytes, dtype=torch.uint8, device=self.device)
                dist.all_gather_into_tensor(everyone, mine)
                # (rank, array) -> (array, rank) on the device, so that the host side is a view of the pinned buffers
                everyone = everyone.view(world, nbytes)
                for key, tail, dtype, at, nb in layout:
                    dev = everyone[:, at:at + nb].contiguous()
                    host["all_" + key] = torch.empty(dev.shape, dtype=torch.uint8, pin_memory=True)
                    host["all_" + key].copy_(dev, non_blocking=True)
                names = ["obs_flags", "window"]
            for k in names:
                src = b[k]
                host[k] = torch.empty(src.shape, dtype=src.dtype, pin_memory=True)
                host[k].copy_(src, non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
        h = {k: v.numpy() for k, v in host.items()}
        d2h = b["means"].numel() * 8 + b["sig"].numel() * 8 + P * 8 + b["obs_flags"].numel()
        if self.return_particles:
            d2h += b["particles"].numel() * 8 + b["weights"].numel() * 8
        if gather is not None:
            out = {key: h["all_" + key].reshape(-1).view(dtype).reshape((world * per,) + tuple(tail))[:ntracks]
                   for key, tail, dtype, at, nb in layout}
            d2h *= world
        else:
            n = h["means"].shape[0]
            out = {"means": h["means"], "sigmas": h["sig"].reshape(n, T, 6, 6) if self.return_covariances else h["sig"],
                   "status": h["status"], "status_time": h["status_time"], "obs_flags": h["obs_flags"]}
            if self.return_particles:
                out["particles"], out["weights"] = h["particles"], h["weights"]
        win = h["window"]
        used = (h["obs_flags"] == 0) & (win[..., 0] > 0)
        self.stats = {
            "plan": {k: getattr(self.plan, k) for k, _ in self.plan._fields_}, "kernel_launches": self.launches,
            "h2d_bytes": int(self.h2d), "d2h_bytes": int(d2h),
            "window_width": win[..., 0][used], "window_height": win[..., 1][used],
        }
        return out

    def final_state(self):
        """What the reference leaves on the Tracker: particles / weights / templates of the last track."""
        b = self.buf
        if int(b["status"][-1]) != 0:  # the last point failed: its buffers stopped at the time of the error
            return None, None, self.templates(self.P - 1)
        final = b["state_b"] if (int(self.last[-1]) & 1) else b["state_a"]
        particles = final[-1].T.contiguous().cpu().numpy()
        if b["final_weights"] is not None:
            weights = b["final_weights"].cpu().numpy()
        else:
            weights = b["weight_state"][-1].cpu().numpy() if b["weight_state"] is not None else np.ones(self.N)
        return particles, weights, self.templates(self.P - 1)

    def templates(self, p: int):
        b = self.buf
        out = []
        for o in range(self.O):
            n_val = int(b["tmpl_nvalues"][p, o])
            if n_val == 0:
                out.append(None)
                continue
            out.append({
                "obs": o, "img": int(self.image_index[self.tmpl_frame[o], o]), "box": b["tmpl_box"][p, o].cpu().numpy(),
                "duv": b["tmpl_duv"][p, o].cpu().numpy(),
                "tile": b["tmpl_tile"][p, o].cpu().numpy().reshape(self.th, self.tw),
                "histogram": (b["tmpl_values"][p, o, :n_val].cpu().numpy(), b["tmpl_quantiles"][p, o, :n_val].cpu().numpy()),
            })
        return out
