"""Raster.viewshed with rings of more cells than the sort holds in shared memory (C = 16 384): the chunked sort, the merge passes
and the sampled horizon search of gb_viewshed.

* Every stored golden of the reference (tests/golden/viewshed.npz) again, with the capacity lowered through the test hook
  GB_VS_RING_CAP, so that their rings take the large-ring path: equal cell for cell.
* DEMs whose rings really exceed C against the oracle (oracle.tracker_oracle.viewshed, pinned bit for bit to the reference by
  test_oracle.py::test_viewshed_vs_reference), computed here: equal cell for cell.
* On the CPU: the work-buffer size and the refusal of more than 2^31 cells before any device work."""
import ctypes as C
import warnings

import numpy as np
import pytest

import helpers
import scenes
from oracle import tracker_oracle as orc

CAP = 16384  # GB_VS_MAX_RING


def ring_numbers(shape, xlim, ylim, origin):
    """Every cell's ring, as the reference numbers them (raster.py:1293-1389; oracle.viewshed)."""
    ny, nx = shape
    x, y = orc.grid_centres(xlim, nx), orc.grid_centres(ylim, ny)
    dx = np.tile(x - origin[0], ny)
    dy = np.repeat(y - origin[1], nx)
    cell = abs((xlim[1] - xlim[0]) / nx)
    return (np.sqrt(dx ** 2 + dy ** 2) * (1 / cell) + 0.5).astype(int)


def run(case, cap=None, monkeypatch=None):
    import glimpse_b200 as gb

    if cap is not None:
        monkeypatch.setenv("GB_VS_RING_CAP", str(cap))
    corr = case["correction"]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return gb.Raster(case["z"], x=case["xlim"], y=case["ylim"]).viewshed(
            case["origin"], correction=dict(radius=corr[0], refraction=corr[1]) if corr else False)


def golden_cases():
    cases = dict(scenes.viewshed_cases())
    cases["large_2000"] = scenes.viewshed_large_case()
    return cases


@pytest.fixture(scope="module")
def goldens():
    return golden_cases(), helpers.load_golden("viewshed")


@pytest.mark.gpu
@pytest.mark.parametrize("cap", [64, 1024])
@pytest.mark.parametrize("name", list(golden_cases()))
def test_forced_capacity_matches_reference(cuda, goldens, monkeypatch, name, cap):
    """The reference's boolean arrays through the large-ring path: rings of more than `cap` cells are sorted in runs of `cap`
    cells and merged, and the ring after one is searched through every k-th abscissa."""
    cases, g = goldens
    case = cases[name]
    ref = np.unpackbits(g[name])[: case["z"].size].reshape(case["z"].shape).astype(bool)
    vis = run(case, cap, monkeypatch)
    assert vis.shape == ref.shape
    assert int((vis != ref).sum()) == 0, f"{int((vis != ref).sum())} of {ref.size} cells differ"


def test_forced_capacity_covers_transitions():
    """The forced runs above see rings over the capacity after smaller ones and smaller ones after them (with NaN cells too),
    and at 1 024 the full-size golden needs three merge passes (rings up to ~6 300 cells)."""
    cases = golden_cases()

    def sizes(name):
        c = cases[name]
        s = np.bincount(ring_numbers(c["z"].shape, c["xlim"], c["ylim"], c["origin"]))
        return s[s > 0]

    for name, cap in (("interior", 64), ("nan_cells", 64), ("big", 64), ("large_2000", 64), ("large_2000", 1024)):
        s = sizes(name)
        up = (s[:-1] <= cap) & (s[1:] > cap)
        down = (s[:-1] > cap) & (s[1:] <= cap)
        assert up.any() and down.any(), (name, cap)
    assert 4 * 1024 < sizes("large_2000").max() <= 8 * 1024


def raised(case, metres):
    ox, oy, oz = case["origin"]
    return dict(case, origin=(ox, oy, oz + metres))


def bumpy(seed, ny, nx, extent, relief, spacing):
    """Seeded terrain of `relief` metres over a square of `extent` metres: bilinear blow-up of noise on a `spacing`-metre grid,
    sampled at the cell centres (cells of extent / nx by extent / ny metres)."""
    from scipy.ndimage import map_coordinates

    rng = np.random.RandomState(seed)
    k = int(extent / spacing) + 2
    coarse = rng.rand(k, k) * relief
    yy = (np.arange(ny) + 0.5) * (extent / ny) / spacing
    xx = (np.arange(nx) + 0.5) * (extent / nx) / spacing
    return map_coordinates(coarse, np.meshgrid(yy, xx, indexing="ij"), order=1)


def stretched(factor, nx, origin=None, holes=False, above=25.0):
    """nx columns of `factor` m by nx * factor rows of 1 m: a square DEM of non-square cells.  Rings are counted in columns, so
    each holds about 2 pi r * factor cells."""
    ny = nx * factor
    ext = float(nx * factor)
    z = bumpy(11 + factor, ny, nx, ext, relief=60.0, spacing=ext / 24)
    if holes:  # NaN patches across the outer (largest) rings, and one just off the eye
        z[ny // 2 + 3000:ny // 2 + 3400, nx // 2 - 40:nx // 2 + 40] = np.nan
        z[ny // 10:ny // 10 + 600, 30:200] = np.nan
        z[ny // 2 - 20:ny // 2 + 20, nx // 2 + 2:nx // 2 + 4] = np.nan
    if origin is None:
        origin = (ext / 2 + 3.3, ext / 2 - 4.1)
    row = min(max(int((ext - origin[1]) / 1.0), 0), ny - 1)
    col = min(max(int(origin[0] / factor), 0), nx - 1)
    eye = float(np.nanmax(z[max(row - 40, 0):row + 40, max(col - 2, 0):col + 3])) + above
    return dict(z=z, xlim=(0.0, ext), ylim=(ext, 0.0), origin=(origin[0], origin[1], eye), correction=None)


LARGE = {
    # 36 M cells, ~400 rings over C (the largest ~18 900): the eye 300 m above the full-size case's
    "square_6000": (lambda: raised(scenes.viewshed_large_case(6000), 270.0), CAP),
    # largest ring ~36 000 cells: more than the sweep's shared memory holds, two merge passes
    "dx16": (lambda: stretched(16, 720), 2 * CAP),
    # largest ring ~84 000 cells: three merge passes, a horizon of ~670 KB in global memory
    "dx64": (lambda: stretched(64, 420), 5 * CAP),
    "dx16_nan": (lambda: stretched(16, 720, holes=True), 2 * CAP),
    # the eye 500 m west of the DEM and 150 m up: every ring is a partial arc, the largest ~17 000 cells
    "dx16_outside": (lambda: stretched(16, 720, origin=(-500.0, 5767.7), above=150.0), CAP),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(LARGE))
def test_large_rings_match_oracle(cuda, name):
    make, covers = LARGE[name]
    case = make()
    rings = ring_numbers(case["z"].shape, case["xlim"], case["ylim"], case["origin"])
    sizes = np.bincount(rings)
    assert sizes.max() > covers, (name, sizes.max())
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        want = orc.viewshed(case["z"], case["xlim"], case["ylim"], case["origin"], case["correction"])
    got = run(case)
    diff = int((got != want).sum())
    assert diff == 0, f"{diff} of {want.size} cells differ"
    # the rings over C say something: they hold visible and hidden cells, some of them both
    big = np.flatnonzero(sizes > CAP)
    vis_in = np.bincount(rings, weights=got.ravel(), minlength=sizes.size)[big]
    assert 0 < vis_in.sum() < sizes[big].sum() and np.any((vis_in > 0) & (vis_in < sizes[big])), name
    if name == "dx16_nan":
        assert np.isnan(case["z"].ravel()[np.isin(rings, big)]).any()


@pytest.mark.gpu
def test_non_square_cells_still_warn(cuda):
    case = stretched(64, 420)
    import glimpse_b200 as gb

    with pytest.warns(UserWarning, match="not square"):
        gb.Raster(case["z"], x=case["xlim"], y=case["ylim"]).viewshed(case["origin"])


def test_work_bytes_linear_without_overflow():
    """64 bytes per cell, 12 per ring and a constant: positive and linear in the number of cells up to 46 340 squared."""
    from glimpse_b200 import _lib

    lib = _lib.load()
    prev = 0
    for side in (1, 100, 2000, 10000, 30000, 46340):
        b = lib.gb_viewshed_work_bytes(side, side, 8)
        assert b > prev
        assert 64 * side * side <= b <= 64 * side * side + 4096, (side, b)
        prev = b
    assert lib.gb_viewshed_work_bytes(46340, 46340, 65540) - lib.gb_viewshed_work_bytes(46340, 46340, 8) <= 12 * 65532 + 1024


def test_more_than_2_31_cells_refused_before_device_work():
    """GB_E_RESOURCE before anything touches the (here bogus) device pointers or the CUDA runtime."""
    from glimpse_b200 import _lib

    lib = _lib.load()
    fake = C.c_void_p(16)
    origin = (C.c_double * 3)(0.0, 0.0, 0.0)
    assert lib.gb_viewshed(fake, 46341, 46341, fake, fake, 1.0, origin, None, 65540, fake, 1 << 62, fake, None) == -3
    assert b"2^31" in lib.gb_last_error()
    assert lib.gb_viewshed(fake, 65536, 32768, fake, fake, 1.0, origin, None, 65540, fake, 1 << 62, fake, None) == -3
