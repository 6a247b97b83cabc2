"""Single-stream drop-in shim on the GPU (SURVEY 8(f)-4).

1. The reference's OWN test programs that stay inside the hot path's boundary (tests/test_golden_pcm.c,
   test_noise_determinism.c, test_floattoshort_parity.c, test_frame_paths.c, test_api.c, test_ecc.c of arancormonk/mbelib-neo),
   compiled unmodified by oracle/Makefile (`make shimtests`, binaries in oracle/_ref/, shipped with the repo snapshot) and
   linked against libmbe-neo-b200shim.so instead of libmbe-neo: they must pass frame by frame on the CUDA path.
2. A frame-by-frame run through the shim's mbe_process<Codec>Frame with a caller-owned mbe_parms triplet against the
   oracle's batch run of the same stream: PCM, parameter bits, error counts and the final triplet."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import mbe_testlib as T
from __graft_entry__ import ROOT

pytestmark = pytest.mark.gpu

SHIM = os.path.join(ROOT, "mbelib-neo_b200", "libmbe-neo-b200shim.so")
REFTESTS = ["test_golden_pcm", "test_noise_determinism", "test_floattoshort_parity", "test_frame_paths", "test_api", "test_ecc",
            "test_params", "test_input_validation"]


@pytest.mark.parametrize("name", REFTESTS)
def test_reference_test_program_passes_on_the_gpu_path(name):
    exe = os.path.join(ROOT, "oracle", "_ref", "shim_" + name)
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/shim_%s not built (needs the reference's sources at build time: MBELIB_NEO_SRC)" % name)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, "%s failed on the shim:\n%s\n%s" % (name, r.stdout[-2000:], r.stderr[-2000:])


def test_golden_pcm_known_answer_through_the_shim():
    """The known answer of the reference's tests/test_golden_pcm.c, stored here, on the shim's GPU path: its fixture frame
    (fill_params) through mbe_synthesizeSpeechf with the thread RNG seeded 0xC0FFEE, then mbe_floattoshort; FNV-1a of the
    float PCM 0x59741032, of the int16 PCM 0x4EDB8636 (the oracle's side is tests/test_oracle_kat.py)."""
    shim = ctypes.CDLL(SHIM)
    vp = ctypes.c_void_p
    shim.mbe_setThreadRngSeed.argtypes = [ctypes.c_uint32]
    shim.mbe_initMbeParms.argtypes = [vp, vp, vp]
    shim.mbe_synthesizeSpeechf.argtypes = [vp, vp, vp]
    shim.mbe_floattoshort.argtypes = [vp, vp]
    cur, prev, enh = (np.zeros(T.PARMS_BYTES, np.uint8) for _ in range(3))
    shim.mbe_initMbeParms(T._ptr(cur), T._ptr(prev), T._ptr(enh))
    f, i = cur.view(np.float32), cur.view(np.int32)
    f[0] = np.float32(0.105)
    i[1] = 36
    for l in range(1, 37):
        i[3 + l] = 1 if l % 4 else 0
        f[60 + l] = np.float32(0.035) + np.float32(0.0015) * np.float32(l)
        f[174 + l] = np.float32(l) * np.float32(0.03)
        f[231 + l] = np.float32(l) * np.float32(0.02)
    prev[:] = cur
    shim.mbe_setThreadRngSeed(0xC0FFEE)
    out = np.zeros(160, np.float32)
    pcm = np.zeros(160, np.int16)
    shim.mbe_synthesizeSpeechf(T._ptr(out), T._ptr(cur), T._ptr(prev))
    shim.mbe_floattoshort(T._ptr(out), T._ptr(pcm))
    assert T.fnv1a32(out.tobytes()) == 0x59741032
    assert T.fnv1a32(pcm.tobytes()) == 0x4EDB8636


class Result(ctypes.Structure):
    _fields_ = [("c0_errors", ctypes.c_int), ("protected_errors", ctypes.c_int), ("c4_errors", ctypes.c_int),
                ("total_errors", ctypes.c_int), ("flags", ctypes.c_uint)]


FRAME_FN = {0: "mbe_processImbe7200x4400", 1: "mbe_processImbe7100x4400", 2: "mbe_processAmbe3600x2400",
            3: "mbe_processAmbe3600x2450"}


@pytest.mark.parametrize("codec,soft", [(0, 0), (1, 0), (2, 0), (3, 0), (0, 1), (3, 1)])
def test_frame_by_frame_through_the_shim_equals_the_oracle(codec, soft):
    shim = ctypes.CDLL(SHIM)
    F = 24
    seed = 0xC0FFEE + 7
    hard = T.random_hard_frames(codec, 1, F, 0x51A + codec)
    frames = T.soften(hard, np.random.default_rng(5), flip_p=0.0, rel_ok=0) if soft else hard
    if soft:  # random reliabilities
        frames[..., 1] = np.random.default_rng(6).integers(0, 256, size=frames[..., 1].shape)
    want = T.run_cpu(T.load_oracle().mbo_run, codec, soft, frames, np.array([seed], np.uint32))
    vp = ctypes.c_void_p
    shim.mbe_setThreadRngSeed.argtypes = [ctypes.c_uint32]
    shim.mbe_initMbeParms.argtypes = [vp, vp, vp]
    fn = getattr(shim, FRAME_FN[codec] + ("SoftFrame" if soft else "Frame"))
    fnf = getattr(shim, FRAME_FN[codec] + ("SoftFramef" if soft else "Framef"))
    fn.argtypes = fnf.argtypes = [vp] * 7
    trip = np.zeros((2, 3, T.PARMS_BYTES), np.uint8)   # one triplet per output flavour
    pcm = np.zeros((F, 160), np.int16)
    pcmf = np.zeros((F, 160), np.float32)
    bits = np.zeros((F, T.PARAM_BITS[codec]), np.uint8)
    total = np.zeros(F, np.int32)
    for k, (f_, out) in enumerate(((fn, pcm), (fnf, pcmf))):
        shim.mbe_setThreadRngSeed(seed)
        shim.mbe_initMbeParms(trip[k, 0].ctypes.data, trip[k, 1].ctypes.data, trip[k, 2].ctypes.data)
        for f in range(F):
            r = Result()
            fr = np.ascontiguousarray(frames[0, f])
            rc = f_(out[f].ctypes.data, ctypes.addressof(r), fr.ctypes.data, bits[f].ctypes.data, trip[k, 0].ctypes.data,
                    trip[k, 1].ctypes.data, trip[k, 2].ctypes.data)
            assert rc == r.total_errors >= 0
            total[f] = rc
    assert np.array_equal(bits, want["bits"][0])
    assert np.array_equal(total, want["results"][0, :, 4])
    d = np.abs(pcm.astype(np.int32) - want["pcm"][0].astype(np.int32))
    assert d.max() <= 2 and (d == 0).mean() >= 0.9999   # the north star's PCM tolerance (measured: exact)
    assert np.array_equal(pcmf.view(np.uint32), want["pcmf"][0].view(np.uint32))
    final = want["state"][0].reshape(3, T.PARMS_BYTES)
    assert np.array_equal(trip[0], final) and np.array_equal(trip[1], final)


def test_two_threads_keep_their_own_rng_state():
    """The reference keeps its RNG in thread-local storage (mbelib.h:28-30); the shim does too.  Two host threads decode
    different streams through the shim at the same time (seeded differently, unvoiced-heavy random frames, so the noise
    generator matters) and each must equal the oracle's run of its own stream."""
    import threading
    shim = ctypes.CDLL(SHIM)
    vp = ctypes.c_void_p
    shim.mbe_setThreadRngSeed.argtypes = [ctypes.c_uint32]
    shim.mbe_initMbeParms.argtypes = [vp, vp, vp]
    F = 30
    jobs = [(3, 0xAAA1), (0, 0xBBB2)]
    out = {}

    def work(codec, seed):
        fn = getattr(shim, FRAME_FN[codec] + "Frame")
        fn.argtypes = [vp] * 7
        frames = T.random_hard_frames(codec, 1, F, seed)
        trip = np.zeros((3, T.PARMS_BYTES), np.uint8)
        pcm = np.zeros((F, 160), np.int16)
        bits = np.zeros(T.PARAM_BITS[codec], np.uint8)
        shim.mbe_setThreadRngSeed(seed)
        shim.mbe_initMbeParms(trip[0].ctypes.data, trip[1].ctypes.data, trip[2].ctypes.data)
        for f in range(F):
            fr = np.ascontiguousarray(frames[0, f])
            rc = fn(pcm[f].ctypes.data, None, fr.ctypes.data, bits.ctypes.data, trip[0].ctypes.data, trip[1].ctypes.data,
                    trip[2].ctypes.data)
            assert rc >= 0
        out[codec] = (frames, pcm)

    th = [threading.Thread(target=work, args=j) for j in jobs]
    for t in th:
        t.start()
    for t in th:
        t.join()
    for codec, seed in jobs:
        frames, pcm = out[codec]
        want = T.run_cpu(T.load_oracle().mbo_run, codec, 0, frames, np.array([seed], np.uint32))
        assert np.array_equal(pcm, want["pcm"][0]), T.CODEC_NAMES[codec]


def test_sixteen_threads_decode_side_by_side():
    """The reference is re-entrant per stream (mbelib.h:28-30).  Every calling thread of the shim owns its context (no lock
    in the shim), so 16 threads decoding 16 different streams at once each equal the oracle's run of their own stream.
    A frame through the shim is one mbe_b200_single_frame call (one upload, three kernel launches, one download, one
    synchronisation); the CUDA driver still serialises the runtime calls of one process on its own locks, so 16 threads decode
    ~3x, not 16x, faster than one (measured: 17.8 k frames/s alone, 53 k frames/s with 16 threads) - the batched C-ABI is the
    throughput path, the shim is the compatibility path (DESIGN 8-4).  Timing is printed, not asserted: a thread's frame loop
    overlaps the other threads' context creation (device allocations serialise the whole process), which moves the slowest
    thread's time between 12 ms and 250 ms from run to run."""
    import threading
    import time
    shim = ctypes.CDLL(SHIM)
    vp = ctypes.c_void_p
    shim.mbe_setThreadRngSeed.argtypes = [ctypes.c_uint32]
    shim.mbe_initMbeParms.argtypes = [vp, vp, vp]
    codec, F, N = 3, 40, 16
    fn = getattr(shim, FRAME_FN[codec] + "Frame")
    fn.argtypes = [vp] * 7
    out = {}

    def work(i):
        seed = 0x5EED0 + i
        frames = T.random_hard_frames(codec, 1, F, seed)
        trip = np.zeros((3, T.PARMS_BYTES), np.uint8)
        pcm = np.zeros((F, 160), np.int16)
        bits = np.zeros(T.PARAM_BITS[codec], np.uint8)
        shim.mbe_setThreadRngSeed(seed)
        shim.mbe_initMbeParms(trip[0].ctypes.data, trip[1].ctypes.data, trip[2].ctypes.data)
        t0 = time.perf_counter()
        for f in range(F):
            fr = np.ascontiguousarray(frames[0, f])
            rc = fn(pcm[f].ctypes.data, None, fr.ctypes.data, bits.ctypes.data, trip[0].ctypes.data, trip[1].ctypes.data,
                    trip[2].ctypes.data)
            assert rc >= 0
        out[i] = (frames, pcm, seed, time.perf_counter() - t0)

    work(100)                                  # warm-up (context creation, first launches) and the single-thread time
    work(101)
    t_one = out[101][3]
    th = [threading.Thread(target=work, args=(i,)) for i in range(N)]
    t0 = time.perf_counter()
    for t in th:
        t.start()
    for t in th:
        t.join()
    t_all = time.perf_counter() - t0
    for i in range(N):
        frames, pcm, seed, _ = out[i]
        want = T.run_cpu(T.load_oracle().mbo_run, codec, 0, frames, np.array([seed], np.uint32))
        assert np.array_equal(pcm, want["pcm"][0]), i
    # includes 16 context creations; a serialised shim would need >= 16 x t_one for the frames alone
    print("one thread %.3f s, 16 threads %.3f s (%.1fx one)" % (t_one, t_all, t_all / t_one))
    steady = max(out[i][3] for i in range(N))
    print("slowest thread's %d frames: %.4f s (one thread alone: %.4f s = %.0f frames/s); %d threads: %.0f frames/s in steady state" % (
        F, steady, t_one, F / t_one, N, N * F / steady))
