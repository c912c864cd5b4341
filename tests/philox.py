"""The device draws of ``rng='philox'`` restated on the host, read back from the device, and replayed to the CPU oracle.

Keying as ``glimpse_b200/csrc/motion.cuh`` states it: Philox4x32-10 (Salmon et al., SC'11) with key
``(seed & 0xffffffff, seed >> 32)`` and counter ``(particle, time, point & 0xffffffff, (point >> 32) << 8 | stream)``.
Streams: 0 and 1 = the six normals of a point's first frame (at time ``first``), 2 = the three normals of every later step,
3 = the systematic resampler's uniform (particle word ``0xffffffff``), 4 = one uniform per particle for the stratified,
choice and residual resamplers.
"""
import ctypes as C

import numpy as np

MASK32 = np.uint64(0xFFFFFFFF)
M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
SYSTEMATIC_PARTICLE = 0xFFFFFFFF


def philox4x32_10(counter, key):
    """Philox4x32-10: ``counter`` = four arrays (or numbers) of 32-bit words, ``key`` = two; broadcast together.  Returns
    the four output words as uint64 arrays (values below 2^32)."""
    c = [np.asarray(x, dtype=np.uint64) & MASK32 for x in counter]
    c = list(np.broadcast_arrays(*c, *[np.asarray(k, dtype=np.uint64) for k in key]))
    k0, k1 = c[4] & MASK32, c[5] & MASK32
    c = c[:4]
    for _ in range(10):
        p0, p1 = M0 * c[0], M1 * c[2]  # (products of two 32-bit words fit in 64 bits)
        hi0, lo0 = p0 >> np.uint64(32), p0 & MASK32
        hi1, lo1 = p1 >> np.uint64(32), p1 & MASK32
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
        k0, k1 = (k0 + W0) & MASK32, (k1 + W1) & MASK32
    return c


def counter(particle, time, point, stream):
    point = np.asarray(point, dtype=np.uint64)
    return (particle, time, point & MASK32, ((point >> np.uint64(32)) << np.uint64(8)) | np.uint64(stream))


def key(seed):
    seed = np.uint64(seed)
    return seed & MASK32, seed >> np.uint64(32)


def words(seed, point, time, particle, stream):
    """The four words the device draws for (point, time, particle) of ``stream``."""
    return philox4x32_10(counter(particle, time, point, stream), key(seed))


def uniform53(w0, w1):
    """[0, 1) with 53 random bits from two words, as NumPy's legacy ``random_sample`` builds it from two MT19937 outputs."""
    bits = ((np.asarray(w0, dtype=np.uint64) >> np.uint64(5)) << np.uint64(26)) | (np.asarray(w1, dtype=np.uint64) >> np.uint64(6))
    return bits.astype(np.float64) / 9007199254740992.0


def uniform(seed, point, time):
    """The systematic resampler's uniform of (point, time)."""
    r = words(seed, point, time, SYSTEMATIC_PARTICLE, 3)
    return uniform53(r[0], r[1])


def uniform_particle(seed, point, time, particle):
    """The per-particle uniform (stratified, choice, residual) of (point, time, particle)."""
    r = words(seed, point, time, particle, 4)
    return uniform53(r[0], r[1])


def box_muller64(r):
    """Float64 Box-Muller of the four words ``r`` in the device's construction (u = (w + 1/2) 2^-32 in (0, 1), angle =
    2 pi (w >> 8) 2^-24): the accuracy reference of the device's float32 normals.  Returns (n, 3)."""
    u0 = (r[0].astype(np.float64) + 0.5) * 2.0 ** -32
    u1 = (r[2].astype(np.float64) + 0.5) * 2.0 ** -32
    a0 = 2 * np.pi * (r[1] >> np.uint64(8)).astype(np.float64) * 2.0 ** -24
    a1 = 2 * np.pi * (r[3] >> np.uint64(8)).astype(np.float64) * 2.0 ** -24
    rad0, rad1 = np.sqrt(-2 * np.log(u0)), np.sqrt(-2 * np.log(u1))
    return np.stack([rad0 * np.cos(a0), rad0 * np.sin(a0), rad1 * np.cos(a1)], axis=-1)


# ------------------------------------------------------------------------------------------------ the device's draws
def read(torch, kind, seed, point, time, first, n, stream=0):
    """``gb_philox_draws`` into a fresh device tensor, returned on the host: uint32 (n, 4) words, float64 (n, 3) normals or
    float64 (n,) uniforms."""
    from glimpse_b200 import _lib

    lib = _lib.load()
    shape, dtype = {_lib.GB_DRAW_WORDS: ((n, 4), torch.int32), _lib.GB_DRAW_NORMALS: ((n, 3), torch.float64)}.get(
        kind, ((n,), torch.float64))
    out = torch.empty(shape, dtype=dtype, device="cuda")
    _lib.check(lib.gb_philox_draws(int(seed) % (1 << 64), int(point), int(time) & 0xFFFFFFFF, int(first) & 0xFFFFFFFF, int(n),
                                   int(kind), int(stream), out.data_ptr(), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    host = out.cpu().numpy()
    return host.view(np.uint32) if kind == _lib.GB_DRAW_WORDS else host


def device_draws(seed, global_points, first, last, N, tangent, method):
    """The draws a ``rng='philox'`` track with ``seed`` takes, read from the device, in the layout of
    ``session.reference_order_draws`` (the ``draws`` of a Session): init (P, N, 6) from streams 0 and 1 at time ``first[p]``
    (tangent models: column 5 unused, 0); step (P, S, N, 3) from stream 2 at times first + 1 ... last; unif (P, S) from
    stream 3 for the systematic resampler, (P, S, N) from stream 4 for the others.  ``global_points[p]`` = the point index
    the device keys row p by (its row in the whole track)."""
    import torch

    from glimpse_b200 import _lib

    P = len(global_points)
    steps = np.asarray(last) - np.asarray(first)
    S = max(int(steps.max()) if P else 0, 1)
    per_particle = method != "systematic"
    init = np.zeros((P, N, 6))
    step = np.zeros((P, S, N, 3))
    unif = np.zeros((P, S, N) if per_particle else (P, S))
    for p, g in enumerate(global_points):
        f = int(first[p])
        init[p, :, 0:3] = read(torch, _lib.GB_DRAW_NORMALS, seed, g, f, 0, N, stream=0)
        init[p, :, 3:6] = read(torch, _lib.GB_DRAW_NORMALS, seed, g, f, 0, N, stream=1)
        if tangent[p]:
            init[p, :, 5] = 0.0
        n_steps = int(steps[p])
        for k in range(n_steps):
            step[p, k] = read(torch, _lib.GB_DRAW_NORMALS, seed, g, f + 1 + k, 0, N, stream=2)
            if per_particle:
                unif[p, k] = read(torch, _lib.GB_DRAW_UNIFORM_PARTICLE, seed, g, f + 1 + k, 0, N)
        if not per_particle and n_steps:
            unif[p, :n_steps] = read(torch, _lib.GB_DRAW_UNIFORM, seed, g, f + 1, 0, n_steps)
    return init, step, unif


class replay:
    """``randn`` / ``random`` for ``oracle.tracker_oracle.track`` that hand out (init, step, unif) in the reference's call
    order: per point randn(n,2), randn(n), randn(n,3) (tangent models: randn(n,2)); per update randn(n,3) (tangent:
    randn(n,2), randn(n)), then random() for the systematic resampler, random(n) for stratified and choice, random(m) for
    residual (the first m <= n of that update's row).  ``steps[p]`` = number of updates of point p, ``method`` = the resampler.
    A call out of that order raises AssertionError; ``done`` tells whether every draw was handed out."""

    def __init__(self, init, step, unif, steps, tangent, method):
        assert (unif.ndim == 2) == (method == "systematic"), "systematic: unif (P, S); the other resamplers: (P, S, N)"
        self._queue = self._order(init, step, unif, steps, tangent, method)
        self._next = next(self._queue, None)

    @staticmethod
    def _order(init, step, unif, steps, tangent, method):
        N = init.shape[1]
        for p in range(init.shape[0]):
            yield "randn", (N, 2), init[p, :, 0:2]
            yield "randn", (N,), init[p, :, 2]
            yield ("randn", (N, 2), init[p, :, 3:5]) if tangent[p] else ("randn", (N, 3), init[p, :, 3:6])
            for k in range(int(steps[p])):
                if tangent[p]:
                    yield "randn", (N, 2), step[p, k, :, 0:2]
                    yield "randn", (N,), step[p, k, :, 2]
                else:
                    yield "randn", (N, 3), step[p, k]
                if method == "systematic":
                    yield "random", (), unif[p, k]
                elif method == "residual":
                    yield "random", None, unif[p, k]  # random(m), m <= N
                else:
                    yield "random", (N,), unif[p, k]

    def _take(self, what, shape):
        assert self._next is not None, f"{what}{shape}: every draw was already handed out"
        kind, want, values = self._next
        assert kind == what, f"{what}{shape} called where the reference calls {kind}{want}"
        if want is None:  # residual: the first m of a row
            assert len(shape) == 1 and shape[0] <= len(values), f"random{shape} called for a row of {len(values)} uniforms"
            out = np.array(values[:shape[0]])
        else:
            assert shape == want, f"{what}{shape} called where the reference calls {kind}{want}"
            out = np.array(values) if shape else float(values)
        self._next = next(self._queue, None)
        return out

    def randn(self, *shape):
        return self._take("randn", tuple(shape))

    def random(self, size=None):
        return self._take("random", () if size is None else tuple(np.atleast_1d(size).tolist()))

    @property
    def done(self):
        return self._next is None
