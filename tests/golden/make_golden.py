#!/usr/bin/env python
"""Generates tests/golden/*.npz from the UNMODIFIED reference compiled by oracle/Makefile (oracle/_ref/libref_bench.so,
Release flags = the parity build of SURVEY 8(c)).  Needs the reference's sources once, to build
oracle/_ref:

    MBELIB_NEO_SRC=<checkout of the reference> make -C oracle ref && python tests/golden/make_golden.py

One file per codec and input kind: seeded inputs (random bits = repeats / mutes / re-initialisation; valid frames of held and
changing parameters = stable pitch, interpolated harmonics; valid frames with flipped bits; AMBE tone / erasure signatures) and
what the reference returns for them through mbe_process<Codec>[Soft]Framef + mbe_floattoshort, frame after frame:
parameter bits, result counters and flags, float PCM (bit patterns), int16 PCM, the final mbe_parms triplets.  The repository
does not hold the reference; tests/test_golden_fixtures.py compares the oracle port (CPU) and both GPU kernel paths with these."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import mbe_testlib as T  # noqa: E402


def frames_for(codec, S, F, seed):
    rng = np.random.default_rng(seed)
    fb = T.FRAME_BITS[codec]
    enc = {0: T.encode_imbe7200_frame, 1: T.encode_imbe7100_frame}.get(codec, T.encode_ambe_frame)
    frames = rng.integers(0, 2, size=(S, F, fb), dtype=np.uint8)       # stream 0 of every four stays random
    for s in range(S):
        if s % 4 == 0:
            continue
        f = 0
        while f < F:
            n = int(min(F - f, rng.integers(1, 7)))
            p = rng.integers(0, 2, size=T.PARAM_BITS[codec], dtype=np.uint8)
            if codec <= 1:
                p[codec] = 0
            elif rng.random() < 0.2:
                p[0:6] = 1
                if rng.random() < 0.5:
                    p[45:49] = 0
            frames[s, f:f + n] = enc(p).reshape(-1)
            if s % 4 == 2:
                frames[s, f:f + n] ^= (rng.random((n, fb)) < 0.04).astype(np.uint8)
            f += n
    return frames


def main():
    ref = T.load_ref()
    if ref is None:
        raise SystemExit("oracle/_ref/libref_bench.so is missing: run `MBELIB_NEO_SRC=<checkout of the reference> make -C oracle ref`")
    for codec in range(4):
        for soft in (0, 1):
            S, F = (8, 32) if not soft else (4, 12)
            frames = frames_for(codec, S, F, 0x601D + 16 * codec + soft)
            if soft:
                frames = T.soften(frames, np.random.default_rng(0x50F7 + codec), flip_p=0.06)
            seeds = T.stream_seeds(S, 0x5EED + codec)
            out = T.run_cpu(ref.ref_bench_run, codec, soft, frames, seeds)
            name = os.path.join(HERE, "%s_%s.npz" % (T.CODEC_NAMES[codec], "soft" if soft else "hard"))
            np.savez_compressed(name, codec=np.int32(codec), soft=np.int32(soft), frames=frames, seeds=seeds, bits=out["bits"],
                                results=out["results"], pcm=out["pcm"], pcmf_bits=out["pcmf"].view(np.uint32), state=out["state"])
            print(name, os.path.getsize(name), "bytes;", S, "streams x", F, "frames; max |pcm|", int(np.abs(out["pcm"]).max()))


if __name__ == "__main__":
    main()
