"""The two kernel paths of the frame entry points (DESIGN 4.5) against each other: the fused kernel and the parameter kernel
+ synthesis kernel pair must agree bit for bit - parameter bits, results, int16 and float PCM, and the final mbe_parms
triplets including the previousUw / noiseOverlap arrays the two kernels of the split path own separately.  (Each path is
also checked against the oracle: tests/test_gpu_parity.py runs every case on both.)"""
import numpy as np
import pytest

import mbe_testlib as T
from __graft_entry__ import load_package

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg():
    return load_package()


@pytest.mark.parametrize("codec", [0, 1, 2, 3])
@pytest.mark.parametrize("soft", [0, 1])
def test_split_equals_fused(pkg, codec, soft):
    S, F = (300, 40) if not soft else (60, 12)
    frames = T.mixed_frames(codec, S, F, 0x5917 + 10 * codec + soft)
    if soft:
        rng = np.random.default_rng(codec)
        frames = T.soften(frames, rng, flip_p=0.05)
    seeds = T.stream_seeds(S, 0x51)
    out = []
    for path in (0, 1):
        dec = pkg.Decoder(max_streams=S, device=0)
        dec.set_kernel_path(path)
        dec.init_streams(0, S, seeds)
        # three launches of different lengths: the state round trip between launches is part of the comparison
        cuts = [(0, 1), (1, F // 2), (F // 2, F)]
        parts = [dec.process_frames(codec, np.ascontiguousarray(frames[:, a:b]), soft=bool(soft), want_float=True) for a, b in cuts]
        out.append((parts, dec.export_state(0, S), dec.export_rng(0, S)))
        dec.close()
    (pa, sa, ra), (pb, sb, rb) = out
    for x, y in zip(pa, pb):
        assert np.array_equal(x["bits"], y["bits"])
        assert np.array_equal(x["results"], y["results"])
        assert np.array_equal(x["pcmf"].view(np.uint32), y["pcmf"].view(np.uint32))
        assert np.array_equal(x["pcm"], y["pcm"])
    assert np.array_equal(sa, sb), "final parameter sets differ (previousUw / noiseOverlap included)"
    assert np.array_equal(ra, rb)


def test_split_descriptor_buffer_ranges(pkg, monkeypatch):
    """A batch whose descriptors exceed the buffer budget is cut into stream ranges inside the call (MBE_B200_DESC_MB is read
    once per process, so this test only checks a batch much larger than one block through both paths: ragged last block,
    stream window in the middle of the pool; tests/test_gpu_knobs.py cuts real ranges under a 1 MiB budget in child
    processes)."""
    codec, S, F = 3, 1000, 9
    frames = T.random_hard_frames(codec, S, F, 0xD5C)
    seeds = T.stream_seeds(S + 50, 7)
    res = []
    for path in (0, 1):
        dec = pkg.Decoder(max_streams=S + 50, device=0)
        dec.set_kernel_path(path)
        dec.init_streams(0, S + 50, seeds)
        got = dec.process_frames(codec, frames, first_stream=37, want_float=True)
        res.append((got, dec.export_state(0, S + 50)))
        dec.close()
    assert np.array_equal(res[0][0]["pcmf"].view(np.uint32), res[1][0]["pcmf"].view(np.uint32))
    assert np.array_equal(res[0][0]["results"], res[1][0]["results"])
    assert np.array_equal(res[0][1], res[1][1])


def test_kernel_timing_and_bank_counters(pkg):
    """mbe_b200_set_kernel_timing / kernel_timing (bench.py's roofline source): per kernel kind launches and device time, and
    the bank kernel's own work counters.  Voice frames of valid AMBE+2 parameters all run the synthesis, so the frame counter
    is exact; the slot counter must lie between one and 112 per synthesised frame; the fused path reports one kind only."""
    codec, S, F = 3, 200, 10
    rng = np.random.default_rng(77)
    frames = np.zeros((S, F, 96), np.uint8)
    for s in range(S):
        for f in range(F):
            p = rng.integers(0, 2, size=49, dtype=np.uint8)
            p[0] = 0                                    # b0 < 64: a voice frame, never a tone / erasure signature
            frames[s, f] = T.encode_ambe_frame(p).reshape(-1)
    dec = pkg.Decoder(max_streams=S, device=0)
    for path in (1, 0):
        dec.set_kernel_path(path)
        dec.init_streams(0, S, T.stream_seeds(S, 1))
        dec.set_kernel_timing(True)
        got = dec.process_frames(codec, frames)
        kinds, work = dec.kernel_timing()
        dec.set_kernel_timing(False)
        assert (got["results"]["status"] >= 0).all()
        if path == 1:
            assert all(kinds[k][1] >= 1 and kinds[k][0] > 0.0 for k in ("parameter", "bank", "unvoiced")), kinds
            muted = int(((got["results"]["flags"] & 0x80) != 0).sum())
            assert S * F - muted <= work["frames"] <= S * F
            assert work["frames"] <= work["slots"] <= 112 * work["frames"]
            assert 0 <= work["interpolated"] <= 7 * work["frames"]
        else:
            assert kinds["parameter"][1] >= 1 and kinds["bank"][1] == 0 and kinds["unvoiced"][1] == 0
            assert work == dict(slots=0, interpolated=0, frames=0)
    with pytest.raises(pkg.MbeB200Error):
        dec.set_kernel_path(2)
    dec.close()


# (codec, input): hard and soft input for every codec through the host pipeline, and hard input through one device-resident
# call large enough that every bank warp walks at least 64 frames (its 32-frame window fills and moves, DESIGN 4.5)
FUZZ_CASES = [pytest.param(c, s, id="%d-%s" % (c, s)) for s in ("hard", "soft") for c in (0, 1, 2, 3)] + \
             [pytest.param(c, "dev", id="%d-dev" % c) for c in (0, 3)]


@pytest.mark.parametrize("codec,mode", FUZZ_CASES)
def test_state_machine_fuzz_against_the_oracle(pkg, codec, mode):
    """Differential fuzz of the frame state machines on the default (multi-kernel) path: 4096 streams x 24 frames per codec,
    every frame drawn at random from {random bits, a fresh valid frame, the previous valid frame held, a valid frame with
    1-8 % flipped bits, an AMBE tone / erasure signature, a frame with a non-binary bit}, so that repeats, headroom resets,
    mutes, re-initialisation, erasures, replays and tones follow each other in every order - which is what the descriptor's
    previousUw op codes have to replay exactly.  Everything against the oracle: bits, results, int16 / float PCM, final
    triplets.  Soft-decision input: the same mixture with seeded flips and reliabilities (fewer streams: the oracle's
    exhaustive soft decoders are slow), decoded in three launches of different lengths.  Device-resident: hard input, as
    many streams as give 64 frames to each warp of the resident bank grid, in one process_frames_dev call."""
    soft = int(mode == "soft")
    rng = np.random.default_rng(0xF022 + codec + 16 * soft + 32 * (mode == "dev"))
    S, F = (4096, 24) if mode == "hard" else (384, 18) if soft else (0, 24)
    if mode == "dev":
        import torch
        bank_warps = torch.cuda.get_device_properties(0).multi_processor_count * T.BANK_WARPS_PER_SM
        S = -(-64 * bank_warps // F // 64) * 64
    fb, pb = T.FRAME_BITS[codec], T.PARAM_BITS[codec]
    enc = {0: T.encode_imbe7200_frame, 1: T.encode_imbe7100_frame}.get(codec, T.encode_ambe_frame)
    P = 96
    pool = np.zeros((P, fb), np.uint8)
    for i in range(P):
        p = rng.integers(0, 2, size=pb, dtype=np.uint8)
        if codec <= 1:
            p[codec] = 0
        elif i % 6 == 0:
            p[0:6] = 1                      # tone / erasure signatures
            if i % 12 == 0:
                p[45:49] = 0
        pool[i] = enc(p).reshape(-1)
    kind = rng.choice(6, size=(S, F), p=[0.22, 0.30, 0.22, 0.18, 0.06, 0.02])
    pick = rng.integers(0, P, size=(S, F))
    frames = np.zeros((S, F, fb), np.uint8)
    last = pool[pick[:, 0]]
    for f in range(F):
        k = kind[:, f]
        fresh = pool[pick[:, f]]
        cur = np.where((k == 2)[:, None], last, fresh)                 # held frame
        last = np.where(((k == 1) | (k == 2) | (k == 3))[:, None], cur, last)
        noisy = cur ^ (rng.random((S, fb)) < rng.uniform(0.01, 0.08, size=(S, 1))).astype(np.uint8)
        rnd = rng.integers(0, 2, size=(S, fb), dtype=np.uint8)
        out = np.where((k == 0)[:, None], rnd, np.where((k == 3)[:, None], noisy, cur))
        sig = pool[(pick[:, f] // 6) * 6 % P]                          # a signature frame (AMBE) / a valid frame (IMBE)
        out = np.where((k == 4)[:, None], sig, out)
        bad = out.copy()
        bad[:, 7] = 2
        frames[:, f] = np.where((k == 5)[:, None], bad, out)
    seeds = T.stream_seeds(S, 0xF0 + codec)
    if soft:
        frames = T.soften(frames, rng, flip_p=0.03)
        frames[..., 0] = np.where(kind[..., None] == 5, np.where(np.arange(fb) == 7, 2, frames[..., 0]), frames[..., 0])
    want = T.run_cpu(T.load_oracle().mbo_run, codec, soft, frames, seeds, n_threads=16)
    dec = pkg.Decoder(max_streams=S, device=0)
    dec.set_kernel_path(1)
    dec.init_streams(0, S, seeds)
    if soft:
        parts = [dec.process_frames(codec, np.ascontiguousarray(frames[:, a:b]), soft=True, want_float=True)
                 for a, b in ((0, 1), (1, 7), (7, F))]
        got = {k: np.concatenate([p[k] for p in parts], axis=1) for k in ("bits", "results", "pcm", "pcmf")}
    elif mode == "dev":
        d_frames = torch.from_numpy(frames).to("cuda:0")
        d = dict(pcm=torch.empty((S, F, 160), dtype=torch.int16, device="cuda:0"),
                 pcmf=torch.empty((S, F, 160), dtype=torch.float32, device="cuda:0"),
                 results=torch.empty((S, F, 6), dtype=torch.int32, device="cuda:0"),
                 bits=torch.empty((S, F, pb), dtype=torch.uint8, device="cuda:0"))
        torch.cuda.synchronize()
        dec.set_kernel_timing(True)
        dec.process_frames_dev(codec, 0, 0, S, F, d_frames.data_ptr(), d["pcm"].data_ptr(), d["pcmf"].data_ptr(),
                               d["results"].data_ptr(), d["bits"].data_ptr())
        torch.cuda.synchronize()
        _, launches = T.counters(dec)
        dec.set_kernel_timing(False)
        assert launches[1] == 1 and S * F >= 64 * bank_warps
        got = {k: v.cpu().numpy() for k, v in d.items()}
        got["results"] = got["results"].view(pkg.RESULT_DTYPE)[..., 0]
    else:
        got = dec.process_frames(codec, frames, want_float=True)
    res = got["results"]
    assert np.array_equal(res["status"], want["results"][..., 0])
    ok = want["results"][..., 0] >= 0
    assert np.array_equal(got["bits"][ok], want["bits"][ok])
    assert np.array_equal(res["total_errors"][ok], want["results"][..., 4][ok])
    assert np.array_equal(res["flags"][ok].astype(np.int64), want["results"][..., 5][ok].astype(np.int64) & 0xffffffff)
    assert np.array_equal(got["pcmf"].view(np.uint32), want["pcmf"].view(np.uint32))
    assert np.array_equal(got["pcm"], want["pcm"])
    assert np.array_equal(dec.export_state(0, S), want["state"])
    flags = res["flags"][ok]
    print(T.CODEC_NAMES[codec], "frames", int(ok.sum()), "rejected", int((~ok).sum()), "repeat", int((flags & 0x40 != 0).sum()),
          "mute", int((flags & 0x80 != 0).sum()), "tone", int((flags & 0x10 != 0).sum()), "erasure", int((flags & 0x20 != 0).sum()))
    dec.close()
