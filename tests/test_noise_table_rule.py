"""The rule behind the unvoiced kernel's noise spectrum table (mbe_split.cuh), checked on the CPU against a plain LCG
x -> (171 x + 11213) mod 53125: the backward-jump constants (DevTables::uvBA / uvBC = LCG^(53125 - 96 + k)) give the 96
states before a generator state, and the reference's noise generator (the oracle's make_noise) always leaves a natural pair
- overlap word k = LCG^(k - 96)(seed) - so that the next frame of a stream that has left its cold start takes its
spectrum from the table."""
import ctypes

import numpy as np

import mbe_testlib as T

M = 53125


def lcg(x):
    return (171 * x + 11213) % M


def jump(k):
    """(a, c) with LCG^k(x) = (a x + c) mod M, as build_tables computes them"""
    a, c = 1, 0
    for _ in range(k):
        a, c = (171 * a) % M, (171 * c + 11213) % M
    return a, c


BACK = [jump(M - 96 + k) for k in range(96)]


def natural_overlap(sc):
    return [(a * sc + c) % M for a, c in BACK]


def test_full_period():
    x, seen = 0, set()
    for _ in range(M):
        seen.add(x)
        x = lcg(x)
    assert x == 0 and len(seen) == M


def test_backward_jump_constants():
    """the products of the kernel's 32-bit arithmetic do not overflow, and LCG^(96 - k) of overlap word k is sc again"""
    assert all(a * (M - 1) + c < 2 ** 32 for a, c in BACK)
    rng = np.random.default_rng(5)
    for sc in [0, 1, M - 1] + [int(v) for v in rng.integers(0, M, 200)]:
        ov = natural_overlap(sc)
        for k, w in enumerate(ov):
            x = w
            for _ in range(96 - k):
                x = lcg(x)
            assert x == sc
        assert all(lcg(ov[k]) == ov[k + 1] for k in range(95)) and lcg(ov[95]) == sc


def test_reference_noise_generator_leaves_natural_pairs():
    """make_noise (mbe_unvoiced_fft.c, the oracle's mbo_noise_with_overlap) from any warm state: the seed it leaves and the
    overlap it leaves are a natural pair, so whatever overlap a frame imports, the frame after it hits"""
    o = T.load_oracle()
    vp = ctypes.c_void_p
    o.mbo_noise_with_overlap.argtypes = [vp, vp, vp, vp]
    o.mbo_rng_default.argtypes = [vp]
    rng = np.zeros(4, np.uint32)
    o.mbo_rng_default(T._ptr(rng))
    gen = np.random.default_rng(11)
    for trial in range(300):
        seed = np.array([gen.integers(0, 2 * M) + (0.5 if trial % 3 == 0 else 0.0)], np.float32)
        ov = gen.integers(0, M, 96).astype(np.float32)
        buf = np.zeros(256, np.float32)
        o.mbo_noise_with_overlap(T._ptr(buf), T._ptr(seed), T._ptr(ov), T._ptr(rng))
        sc = int(seed[0])
        assert float(sc) == seed[0] and 0 <= sc < M
        assert [int(v) for v in ov] == natural_overlap(sc)
        assert np.array_equal(ov.view(np.uint32), np.array(natural_overlap(sc), np.float32).view(np.uint32))
