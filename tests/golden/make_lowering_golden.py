"""Stored host-side C-ABI tables for the lowering tests of tests/test_host.py.

    python tests/golden/make_lowering_golden.py   ->  tests/golden/lowering.npz

The tables are this package's lowering of the scenes in ``helpers.lowering_scene`` / ``helpers.raster_frames_scene``.
Where the unmodified reference can be imported (``oracle/ref_shim.py``), the script lowers the reference's objects too
and writes nothing unless they give the same bytes; the tests make the same comparison whenever the reference is there.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import glimpse_b200 as gb  # noqa: E402
import helpers  # noqa: E402
from oracle import ref_shim  # noqa: E402

KINDS = ("cartesian", "cylindrical", "tangent_cartesian", "tangent_cylindrical")

apis = [gb] + ([ref_shim.import_reference()] if ref_shim.available() else [])
out = {}
for name, scene, lower in [(kind, helpers.lowering_scene(kind), helpers.lowered_tables) for kind in KINDS] + \
                          [("raster", helpers.raster_frames_scene(), helpers.raster_frame_results)]:
    results = [lower(scene, api) for api in apis]
    for other in results[1:]:
        assert sorted(other) == sorted(results[0]), name
        for key, value in results[0].items():
            np.testing.assert_array_equal(other[key], value, err_msg=f"{name}.{key}: the reference lowers differently")
    out.update({f"{name}.{key}": value for key, value in results[0].items()})
np.savez_compressed(os.path.join(ROOT, "tests", "golden", "lowering.npz"), **out)
print("ok, compared with the reference" if len(apis) > 1 else "ok, reference not importable: not compared",
      {k: v.shape for k, v in out.items()})
