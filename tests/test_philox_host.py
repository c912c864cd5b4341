"""The host restatement of the device generator (tests/philox.py) against published and NumPy's own constructions."""
import numpy as np
import pytest

import philox


@pytest.mark.parametrize("counter,key,expected", [
    # Random123's known-answer vectors for Philox4x32-10 (kat_vectors)
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0), (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
])
def test_philox_known_answers(counter, key, expected):
    assert [int(w) for w in philox.philox4x32_10(counter, key)] == list(expected)


def test_philox_is_vectorised_over_the_counter():
    ctr = np.arange(1000, dtype=np.uint64)
    together = philox.philox4x32_10((ctr, 7, 2 ** 32 - 1, 3), (5, 2 ** 31))
    for i in (0, 1, 999):
        one = philox.philox4x32_10((int(ctr[i]), 7, 2 ** 32 - 1, 3), (5, 2 ** 31))
        assert [int(w[i]) for w in together] == [int(w) for w in one]


def test_keying_splits_point_and_seed_into_words():
    seed, point = (7 << 32) | 11, (3 << 32) | 5
    direct = philox.philox4x32_10((9, 4, 5, (3 << 8) | 2), (11, 7))
    assert [int(w) for w in philox.words(seed, point, 4, 9, 2)] == [int(w) for w in direct]


def test_uniform_is_numpys_random_sample_of_the_same_words():
    """NumPy's legacy random_sample takes two MT19937 outputs a, b and returns ((a >> 5) 2^26 + (b >> 6)) / 2^53; a
    full-range uint32 randint hands out those same outputs one by one."""
    w = np.random.RandomState(2024).randint(0, 2 ** 32, size=2 * 4096, dtype=np.uint32)
    u = np.random.RandomState(2024).random_sample(4096)
    np.testing.assert_array_equal(philox.uniform53(w[0::2], w[1::2]), u)
    assert philox.uniform53(0xFFFFFFFF, 0xFFFFFFFF) == 1.0 - 2.0 ** -53 and philox.uniform53(0, 0) == 0.0


def test_replay_hands_out_draws_in_the_reference_order():
    rng = np.random.RandomState(1)
    P, S, N = 2, 3, 5
    init, step, unif = rng.rand(P, N, 6), rng.rand(P, S, N, 3), rng.rand(P, S)
    r = philox.replay(init, step, unif, steps=[2, 3], tangent=[False, True], method="systematic")
    np.testing.assert_array_equal(r.randn(N, 2), init[0, :, 0:2])
    np.testing.assert_array_equal(r.randn(N), init[0, :, 2])
    np.testing.assert_array_equal(r.randn(N, 3), init[0, :, 3:6])
    for k in range(2):
        np.testing.assert_array_equal(r.randn(N, 3), step[0, k])
        assert r.random() == unif[0, k]
    r.randn(N, 2), r.randn(N)
    np.testing.assert_array_equal(r.randn(N, 2), init[1, :, 3:5])
    with pytest.raises(AssertionError):
        r.randn(N, 3)  # a tangent step draws randn(n, 2) first
    for method in ("stratified", "choice", "residual"):  # a row of N uniforms: all of it, or (residual only) its first m
        r2 = philox.replay(init, step, rng.rand(P, S, N), steps=[1, 0], tangent=[False, False], method=method)
        r2.randn(N, 2), r2.randn(N), r2.randn(N, 3), r2.randn(N, 3)
        assert not r2.done
        with pytest.raises(AssertionError):
            r2.random(N + 1)
        if method != "residual":
            with pytest.raises(AssertionError):
                r2.random(N - 1)
            with pytest.raises(AssertionError):
                r2.random()
        assert len(r2.random(N if method != "residual" else 1)) in (1, N)
    with pytest.raises(AssertionError):
        philox.replay(init, step, unif, steps=[1, 0], tangent=[False, False], method="stratified")
    r3 = philox.replay(init, step, unif[..., None] + np.zeros(N), steps=[1, 0], tangent=[False, False], method="residual")
    r3.randn(N, 2), r3.randn(N), r3.randn(N, 3), r3.randn(N, 3)
    np.testing.assert_array_equal(r3.random(2), unif[0, 0] + np.zeros(2))  # residual: the first m of the row
    r3.randn(N, 2), r3.randn(N), r3.randn(N, 3)
    assert r3.done
    with pytest.raises(AssertionError):
        r3.random()
