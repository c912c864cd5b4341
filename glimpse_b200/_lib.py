"""ctypes binding of ``libglimpse_b200.so`` (the C ABI declared in ``include/glimpse_b200.h``).

There is no CPU fallback: if the shared library is missing, or no CUDA device is present, every
compute entry point raises.  The structures below mirror the header field by field.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libglimpse_b200.so")

GB_MAX_OBS = 8  # observers with a frame at the same time (GB_MAX_OBSERVERS); a call may have any number of observers
GB_ST_MESSAGES = {
    1: (ValueError, "Some particles are on non-visible viewshed cells"),
    2: (ValueError, "Some particles have missing (NaN) values"),
    3: (ValueError, "Some of the sampling coordinates are out of bounds"),
    4: (ValueError, "Some sampling points are outside box"),
    5: (IndexError, "Box extends beyond grid bounds"),
    6: (MemoryError, "Search window larger than the launch plan's surface capacity (template + 191 px per axis in mode='stream'; "
                     "the particle cloud has dispersed)"),
}
GB_OBS_NO_IMAGE, GB_OBS_OUT_OF_FRAME = 1, 2
GB_ST_WINDOW_TOO_LARGE = 6
GB_WINDOW_MARGIN, GB_WINDOW_MARGIN_MAX = 191, 1000  # default / retry capacity of the search windows beyond the template, px
GB_RNG_SUPPLIED, GB_RNG_PHILOX = 0, 1
GB_DRAW_WORDS, GB_DRAW_NORMALS, GB_DRAW_UNIFORM, GB_DRAW_UNIFORM_PARTICLE = 0, 1, 2, 3  # what gb_philox_draws writes
GB_RESAMPLE = {"systematic": 0, "stratified": 1, "choice": 2, "residual": 3}
GB_MODE_STREAM = 1
GB_PIX = {"uint8": 0, "uint16": 1, "float32": 2, "float64": 3}
GB_PLAN_RANKED_FRAMES = 1
GB_PLAN_LARGE_TEMPLATES = 2  # templates above 1024 pixels, up to 128 a side
GB_MAX_TEMPLATE, GB_MAX_TEMPLATE_SIDE = 1024, 128  # template pixels without that flag / largest side with it
GB_HP_MODES = {"reflect": 0, "grid-mirror": 0, "constant": 1, "grid-constant": 1, "nearest": 2, "mirror": 3, "wrap": 4, "grid-wrap": 4}
GB_MOTION_CARTESIAN, GB_MOTION_CYLINDRICAL, GB_MOTION_TANGENT_CARTESIAN, GB_MOTION_TANGENT_CYLINDRICAL = 0, 1, 2, 3


class gb_camera(C.Structure):
    _fields_ = [
        ("R", C.c_double * 9), ("xyz", C.c_double * 3), ("f", C.c_double * 2), ("cc", C.c_double * 2),
        ("k", C.c_double * 6), ("p", C.c_double * 2), ("corr_c1", C.c_double), ("corr_c2", C.c_double),
        ("imgsz", C.c_int32 * 2), ("has_corr", C.c_int32), ("affine", C.c_int32),
    ]


class gb_image(C.Structure):
    _fields_ = [
        ("pixels", C.c_void_p), ("width", C.c_int32), ("height", C.c_int32), ("pitch", C.c_int32), ("nchan", C.c_int32),
        ("dtype", C.c_int32), ("pad_", C.c_int32),
        ("cam", gb_camera),
    ]


class gb_surface(C.Structure):
    _fields_ = [
        ("z", C.c_void_p), ("nx", C.c_int32), ("ny", C.c_int32), ("x0", C.c_double), ("dx", C.c_double),
        ("y0", C.c_double), ("dy", C.c_double), ("xmin", C.c_double), ("xmax", C.c_double), ("ymin", C.c_double),
        ("ymax", C.c_double), ("value", C.c_double),
    ]


class gb_motion(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("dem", C.c_int32), ("dem_sigma", C.c_int32), ("pad_", C.c_int32),
        ("xy", C.c_double * 2), ("xy_sigma", C.c_double * 2), ("v", C.c_double * 3), ("v_sigma", C.c_double * 3),
        ("a", C.c_double * 3), ("a_sigma", C.c_double * 3), ("slope_sigma", C.c_double),
    ]


class gb_plan(C.Structure):
    _fields_ = [
        ("cluster", C.c_int32), ("threads", C.c_int32), ("n_local", C.c_int32), ("particles_in_smem", C.c_int32),
        ("smem_bytes", C.c_int32), ("tile_bytes", C.c_int32), ("max_template", C.c_int32), ("n_slabs", C.c_int32),
        ("slab_bytes", C.c_int64), ("particle_scratch_bytes", C.c_int64), ("scratch_bytes", C.c_int64),
        ("mode", C.c_int32), ("stream_block", C.c_int32), ("stream_nblk", C.c_int32), ("n_observers", C.c_int32),
        ("surf_bytes", C.c_int64), ("stream_batch", C.c_int32), ("stream_slots", C.c_int32),
    ]


class gb_track_desc(C.Structure):
    _fields_ = [
        ("P", C.c_int64), ("N", C.c_int64), ("T", C.c_int32), ("O", C.c_int32), ("tile_w", C.c_int32), ("tile_h", C.c_int32),
        ("images", C.c_void_p), ("images_host", C.c_void_p), ("image_events_host", C.c_void_p), ("image_offset_host", C.c_void_p), ("image_index_host", C.c_void_p),
        ("obs_scale_host", C.c_void_p), ("mask", C.c_void_p), ("first", C.c_void_p), ("last", C.c_void_p),
        ("mask_host", C.c_void_p), ("first_host", C.c_void_p), ("last_host", C.c_void_p),
        ("tau_host", C.c_void_p), ("tau2_host", C.c_void_p),
        ("motion", C.c_void_p), ("surfaces", C.c_void_p), ("n_surfaces", C.c_int32), ("viewshed", C.c_int32),
        ("rng_mode", C.c_int32), ("motion_kinds", C.c_int32), ("seed", C.c_uint64), ("point_offset", C.c_int64),
        ("init_normals", C.c_void_p), ("step_normals", C.c_void_p), ("uniforms", C.c_void_p),
        ("state_a", C.c_void_p), ("state_b", C.c_void_p), ("weight_state", C.c_void_p), ("scratch", C.c_void_p),
        ("tmpl_tile", C.c_void_p), ("tmpl_values", C.c_void_p), ("tmpl_quantiles", C.c_void_p),
        ("tmpl_nvalues", C.c_void_p), ("tmpl_box", C.c_void_p), ("tmpl_duv", C.c_void_p),
        ("means", C.c_void_p), ("sigmas", C.c_void_p), ("covariances", C.c_void_p), ("out_particles", C.c_void_p),
        ("out_weights", C.c_void_p), ("status", C.c_void_p), ("status_time", C.c_void_p), ("obs_flags", C.c_void_p),
        ("window_stats", C.c_void_p),
        ("resample_method", C.c_int32), ("highpass_size", C.c_int32),
        ("interp_rows", C.c_int32), ("interp_cols", C.c_int32),
        ("highpass_mode", C.c_int32), ("highpass_origin", C.c_int32), ("highpass_cval", C.c_double),
        ("highpass_footprint_host", C.c_void_p),
        ("final_weights", C.c_void_p),
        ("plan", gb_plan),
    ]


class gb_stage_io(C.Structure):
    _fields_ = [
        ("force_evolved", C.c_void_p), ("force_weights", C.c_void_p), ("dump_evolved", C.c_void_p),
        ("dump_uv", C.c_void_p), ("dump_box", C.c_void_p), ("dump_search", C.c_void_p), ("dump_sse", C.c_void_p),
        ("dump_sampled", C.c_void_p), ("dump_weights", C.c_void_p), ("dump_indices", C.c_void_p), ("dump_clocks", C.c_void_p), ("dump_cap", C.c_int64),
    ]


# order of gb_struct_size(which)
STRUCTS = (gb_camera, gb_image, gb_surface, gb_motion, gb_plan, gb_track_desc, gb_stage_io)

# name -> (restype, argtypes); every symbol include/glimpse_b200.h declares
SIGNATURES = {
    "gb_version": (C.c_int, []),
    "gb_last_error": (C.c_char_p, []),
    "gb_struct_size": (C.c_int64, [C.c_int32]),
    "gb_sample_surface": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gb_kernel_timing": (C.c_int, [C.c_int32]),
    "gb_kernel_timing_read": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_int64), C.c_int32]),
    "gb_camera_from_vector": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(gb_camera)]),
    "gb_project": (C.c_int, [C.POINTER(gb_camera), C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "gb_project_image": (C.c_int, [C.POINTER(gb_image), C.POINTER(gb_camera), C.c_int32, C.c_void_p, C.c_void_p]),
    "gb_viewshed_work_bytes": (C.c_int64, [C.c_int32, C.c_int32, C.c_int32]),
    "gb_viewshed": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_double, C.POINTER(C.c_double),
                              C.POINTER(C.c_double), C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "gb_jpeg_info": (C.c_int, [C.c_char_p, C.c_int64, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "gb_decode_jpeg": (C.c_int, [C.c_char_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "gb_unproject": (C.c_int, [C.POINTER(gb_camera), C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gb_state_from_rows": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]),
    "gb_state_to_rows": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]),
    "gb_step_plan": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.POINTER(gb_plan)]),
    "gb_step_plan_ex": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(gb_plan)]),
    "gb_track": (C.c_int, [C.POINTER(gb_track_desc), C.c_void_p, C.POINTER(C.c_int64)]),
    "gb_track_step": (C.c_int, [C.POINTER(gb_track_desc), C.c_int32, C.POINTER(gb_stage_io), C.c_void_p]),
    "gb_track_init": (C.c_int, [C.POINTER(gb_track_desc), C.c_int32, C.c_void_p]),
    "gb_evolve": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gb_init_particles": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gb_motion_log_likelihoods": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gb_moments": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gb_philox_draws": (C.c_int, [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int64, C.c_int32, C.c_int32, C.c_void_p,
                                  C.c_void_p]),
}

_lib = None


class LibraryMissing(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the CUDA library (built in-tree by ``__graft_entry__.build()`` / ``glimpse_b200.build``)."""
    global _lib
    if _lib is None:
        path = os.environ.get("GLIMPSE_B200_LIB", LIB_PATH)  # (tuning: a variant built with other -D flags, tools/variants.sh)
        if not os.path.exists(path):
            raise LibraryMissing(
                f"{path} not found: build it with `python -m glimpse_b200.build` (there is no CPU fallback)")
        lib = C.CDLL(path)
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = lib
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().gb_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"glimpse_b200 C-ABI call failed ({rc}): {msg}")


def require_cuda():
    """Return torch after checking a CUDA device is usable (no CPU fallback)."""
    import torch

    if not torch.cuda.is_available():
        raise RuntimeError("glimpse_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch
