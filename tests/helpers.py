"""Test helpers: scene -> oracle inputs, golden loading, reference-order draws."""
import os

import numpy as np

from oracle import tracker_oracle as orc

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)


def oracle_inputs(scene, points=None):
    """(observers, models, taus, image_index) for ``oracle.tracker_oracle.track``."""
    datetimes = scene.datetimes
    observers = [orc.ObserverSpec(o.frames, np.asarray(o.cams), o.sigma) for o in scene.observers]
    image_index = np.full((len(datetimes), len(observers)), -1, dtype=int)
    for j, o in enumerate(scene.observers):
        lookup = {d: i for i, d in enumerate(o.datetimes)}
        for t, d in enumerate(datetimes):
            image_index[t, j] = lookup.get(d, -1)
    unit = scene.time_unit.total_seconds()
    taus = np.array([dt.total_seconds() / unit for dt in np.diff(datetimes)])
    params = dict(scene.motion)
    kind = params.pop("kind")
    names = {"cartesian": ("vxyz", "axyz"), "cylindrical": ("vrthz", "arthz"), "tangent_cartesian": ("vxy", "axy"),
             "tangent_cylindrical": ("vrth", "arth")}[kind]
    pad = lambda x: tuple(x) + (0.0,) * (3 - len(x))  # noqa: E731
    kw = dict(v=pad(params[names[0]]), v_sigma=pad(params[names[0] + "_sigma"]), a=pad(params[names[1]]),
              a_sigma=pad(params[names[1] + "_sigma"]), slope_sigma=params.get("slope_sigma", 0.0))

    def surface(value):
        if isinstance(value, dict):
            return orc.Surface(value["array"], tuple(value["x"]), tuple(value["y"]))
        return orc.Surface(value)

    sel = range(len(scene.points)) if points is None else points
    models = [
        orc.MotionSpec(xy=scene.points[i], n=scene.n_particles, kind=kind, dem=surface(params["dem"]),
                       dem_sigma=surface(params["dem_sigma"]), xy_sigma=params["xy_sigma"], **kw)
        for i in sel
    ]
    return observers, models, taus, image_index


def reference_draws(seed, n_points, n_particles, n_steps_per_point, tangent=False):
    """Draws in the reference's order (SURVEY.md §8c): per point randn(n,2), randn(n), randn(n,3), then per
    later frame randn(n,3) and one random(); the tangent models draw randn(n,2), randn(n), randn(n,2), then per
    frame randn(n,2), randn(n) and one random().  Returns (init (P, n, 6), step (P, S, n, 3), uniforms (P, S))."""
    np.random.seed(seed)
    init = np.zeros((n_points, n_particles, 6))
    step = np.empty((n_points, n_steps_per_point, n_particles, 3))
    unif = np.empty((n_points, n_steps_per_point))
    for p in range(n_points):
        init[p, :, 0:2] = np.random.randn(n_particles, 2)
        init[p, :, 2] = np.random.randn(n_particles)
        if tangent:
            init[p, :, 3:5] = np.random.randn(n_particles, 2)
        else:
            init[p, :, 3:6] = np.random.randn(n_particles, 3)
        for s in range(n_steps_per_point):
            if tangent:
                step[p, s, :, 0:2] = np.random.randn(n_particles, 2)
                step[p, s, :, 2] = np.random.randn(n_particles)
            else:
                step[p, s] = np.random.randn(n_particles, 3)
            unif[p, s] = np.random.random()
    return init, step, unif


def lowering_scene(kind):
    """The scene whose objects ``lowered_tables`` lowers: four points of one motion kind, three jittered frames far from the
    origin of the world, a gridded DEM for the tangent models."""
    import scenes
    from glimpse_b200 import synthetic

    scene = synthetic.nadir_scene(seed=5, n_points=4, n_particles=64, n_frames=3, imgsz=(320, 240), margin_px=90, kind=kind,
                                  jitter_deg=0.05, world_offset=(4.99e5, 6.77e6))
    if kind.startswith("tangent"):
        scenes.add_gridded_dem(scene)
    return scene


def _struct_rows(structs):
    return np.array([np.frombuffer(bytes(s), dtype=np.uint8) for s in structs])


def lowered_tables(scene, api):
    """The host side of the C ABI for ``scene`` built with ``api`` (this package or the reference): the gb_camera of every
    image (one with curvature / refraction corrections), the gb_motion table, the gb_surface table with the cell values of
    its gridded surfaces, and the index of a viewshed raster among the surfaces.  Structs are rows of their bytes."""
    from glimpse_b200 import synthetic
    from glimpse_b200.camera import lower_camera
    from glimpse_b200.session import lower_models

    observers, models = synthetic.build(scene, api)
    observers[0].images[1].cam.correction = {"radius": 6.3781e6, "refraction": 0.13}
    view = api.Raster(np.ones((6, 8)), x=(4.98e5, 5.0e5), y=(6.78e6, 6.76e6))
    table_m, surfaces, vi = lower_models(models, view)
    out = {"cameras": _struct_rows([lower_camera(img.cam) for obs in observers for img in obs.images]),
           "motion": np.frombuffer(table_m.tobytes(), dtype=np.uint8), "surfaces": _struct_rows([s for s, _ in surfaces]),
           "viewshed": np.array(vi)}
    for i, (_, z) in enumerate(surfaces):
        if z is not None:
            out[f"cells{i}"] = np.asarray(z)
    return out


def raster_frames_scene():
    from glimpse_b200 import synthetic

    return synthetic.as_raster_frames(synthetic.nadir_scene(seed=5, n_points=4, n_particles=64, n_frames=3, imgsz=(320, 240),
                                                            margin_px=90, world_offset=(4.99e5, 6.77e6)))


def raster_frame_results(scene, api):
    """An Observer of orthoimages built with ``api``: every frame's affine gb_camera (a row of its bytes) and its answers to
    xyz_to_uv / uv_to_xyz / inbounds at seven fixed points, d, size and read of a fixed box, stacked over the frames."""
    from glimpse_b200 import synthetic
    from glimpse_b200.session import lower_grid_camera

    xyz = np.column_stack((4.99e5 + np.linspace(-40, 40, 7), 6.77e6 + np.linspace(-30, 30, 7), np.zeros(7)))
    out = {k: [] for k in ("camera", "xyz_to_uv", "uv_to_xyz", "inbounds", "d", "size", "read")}
    for img in synthetic.build(scene, api)[0][0].images:
        uv = img.xyz_to_uv(xyz)
        for key, value in (("camera", np.frombuffer(bytes(lower_grid_camera(img)), dtype=np.uint8)), ("xyz_to_uv", uv),
                           ("uv_to_xyz", img.uv_to_xyz(uv)), ("inbounds", img.inbounds(uv - 150)), ("d", img.d),
                           ("size", img.size), ("read", img.read(box=(3, 4, 30, 20)))):
            out[key].append(np.asarray(value))
    return {k: np.stack(v) for k, v in out.items()}


def assert_tables_close(got, want):
    """``lowered_tables`` / ``raster_frame_results`` against stored ones: the same arrays, integers and struct fields of
    integer type equal, floating-point values equal to 1e-12 (relative, or absolute near zero): the stored values come
    from another host, whose libm may round the sines and cosines of a rotation differently in the last bit."""
    from glimpse_b200 import _lib
    from glimpse_b200.session import MOTION_DTYPE

    structs = {"cameras": np.dtype(_lib.gb_camera), "camera": np.dtype(_lib.gb_camera), "surfaces": np.dtype(_lib.gb_surface),
               "motion": MOTION_DTYPE}
    assert sorted(got) == sorted(want), (sorted(got), sorted(want))
    for key, value in got.items():
        ref = np.asarray(want[key])
        assert value.shape == ref.shape, key
        if key in structs:
            value, ref = value.reshape(-1).view(structs[key]), ref.reshape(-1).view(structs[key])
            fields = [(f"{key}.{name}", value[name], ref[name]) for name in structs[key].names]
        else:
            fields = [(key, value, ref)]
        for name, a, b in fields:
            if np.issubdtype(a.dtype, np.floating):
                np.testing.assert_allclose(a, b, rtol=1e-12, atol=1e-12, err_msg=name)
            else:
                np.testing.assert_array_equal(a, b, err_msg=name)


def case_scene(name):
    """(scene, case) of a case of ``scenes.track_cases()`` or ``scenes.shape_cases()``."""
    import scenes
    from glimpse_b200 import synthetic

    case = {**scenes.track_cases(), **scenes.shape_cases()}[name]
    scene = synthetic.nadir_scene(**case["scene_kwargs"])
    if case.get("post"):
        scene = case["post"](scene)
    return scene, case


_SHAPE_CACHE = {}


def shape_golden(name):
    """Full intermediates of a BASELINE-shape case in the key layout of the ``track_*`` goldens, regenerated with the
    oracle and pinned to the compact fixture the unmodified reference produced (``tests/golden/shape_*.npz``): ancestor
    indices, uniform draws, checksums of the evolved particles and weights, means and sigmas must be bit-identical, so
    the regenerated arrays ARE the reference's."""
    import warnings

    if name in _SHAPE_CACHE:
        return _SHAPE_CACHE[name]
    scene, case = case_scene(name)
    small = load_golden(name)
    crc = np.array([int(np.asarray(f, dtype=np.int64).sum()) for o in scene.observers for f in o.frames])
    np.testing.assert_array_equal(crc, small["frame_crc"])
    obs, models, taus, idx = oracle_inputs(scene)
    np.testing.assert_array_equal(idx, small["images"])
    np.random.seed(int(small["seed"]))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        res = orc.track(obs, models, taus, idx, tile_size=scene.tile_size, return_particles=True,
                        return_covariances="covariances" in small, trace=True)
    steps = [s for s in res.trace if "indices" in s]
    assert len(steps) == int(small["n_steps"])
    np.testing.assert_array_equal(np.stack([s["indices"] for s in steps]), small["indices"])
    np.testing.assert_array_equal(np.array([s["u"] for s in steps]), small["u"])
    np.testing.assert_array_equal(np.stack([s["evolved"].sum(axis=0) for s in steps]), small["evolved_sum"])
    np.testing.assert_array_equal(np.array([s["weights"].sum() for s in steps]), small["weights_sum"])
    np.testing.assert_array_equal(np.array([s["weights"].max() for s in steps]), small["weights_max"])
    np.testing.assert_array_equal(res.means, small["means"])
    np.testing.assert_array_equal(res.sigmas, small["covariances"] if "covariances" in small else small["sigmas"])
    np.testing.assert_array_equal(np.nansum(res.particles[:, -1], axis=1), small["final_particles_sum"])
    per = len(steps) // len(models)
    for o, rec in steps[per - 1]["obs"].items():
        np.testing.assert_array_equal(rec["sse"], small[f"last0.obs.{o}.sse"])
        np.testing.assert_array_equal(rec["box"], small[f"last0.obs.{o}.box"])
    g = {k: small[k] for k in small.files}
    g["particles"], g["weights"] = res.particles, res.weights
    for i, s in enumerate(steps):
        for key in ("evolved", "weights", "u", "indices"):
            g[f"step{i}.{key}"] = np.asarray(s[key])
        for o, rec in s.get("obs", {}).items():
            for key, val in rec.items():
                g[f"step{i}.obs.{o}.{key}"] = np.asarray(val)
    assert len(res.templates) == int(small["n_templates"])
    for i, t in enumerate(res.templates):
        np.testing.assert_array_equal(t["box"], small[f"template{i}.box"])
        for key in ("obs", "box", "tile", "values", "quantiles"):
            g[f"template{i}.{key}"] = np.asarray(t[key])
    _SHAPE_CACHE[name] = g
    return g
