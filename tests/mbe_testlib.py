"""Shared helpers for the test-suite: ctypes bindings to the CPU oracle (oracle/libmbe_oracle.so), the
compiled reference (oracle/_ref/*.so, optional) and seeded input generators.

TEST INFRASTRUCTURE ONLY - nothing here is on the product path.
"""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")

IMBE7200, IMBE7100, AMBE2400, AMBE2450 = 0, 1, 2, 3
CODEC_NAMES = {0: "imbe7200x4400", 1: "imbe7100x4400", 2: "ambe3600x2400", 3: "ambe3600x2450"}
FRAME_BITS = {0: 184, 1: 168, 2: 96, 3: 96}
FRAME_SHAPE = {0: (8, 23), 1: (7, 24), 2: (4, 24), 3: (4, 24)}
PARAM_BITS = {0: 88, 1: 88, 2: 49, 3: 49}
PARMS_BYTES = 2604

FLAG_SOFT, FLAG_C0, FLAG_C4, FLAG_TONE, FLAG_ERASURE, FLAG_REPEAT, FLAG_MUTE = 1, 2, 4, 0x10, 0x20, 0x40, 0x80

# field offsets (bytes) inside struct mbe_parameters (include/mbelib-neo/mbelib.h:88-137)
OFF = dict(w0=0, L=4, K=8, Vl=12, Ml=240, log2Ml=468, PHIl=696, PSIl=924, gamma=1152, tonePhase=1156, swn=1160,
           localEnergy=1164, amplitudeThreshold=1168, errorRate=1172, errorCountTotal=1176, errorCount4=1180,
           repeatCount=1184, mutingThreshold=1188, previousUw=1192, noiseSeed=2216, noiseOverlap=2220)


def _build_oracle():
    so = os.path.join(ORACLE_DIR, "libmbe_oracle.so")
    src = os.path.join(ORACLE_DIR, "mbe_oracle.c")
    if (not os.path.exists(so)) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "oracle"], stdout=subprocess.DEVNULL)
    return so


_RUN_ARGS = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
             ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]

_oracle = None
_ref = {}


def load_oracle():
    global _oracle
    if _oracle is None:
        lib = ctypes.CDLL(_build_oracle())
        lib.mbo_run.restype = ctypes.c_double
        lib.mbo_run.argtypes = _RUN_ARGS
        lib.mbo_spectral_amp_enhance.restype = ctypes.c_float
        _oracle = lib
    return _oracle


def ref_available(fast=False):
    name = "libref_bench_fast.so" if fast else "libref_bench.so"
    return os.path.exists(os.path.join(ORACLE_DIR, "_ref", name))


def load_ref(fast=False):
    """The compiled, unmodified reference behind oracle/ref_bench.c (None when oracle/_ref is absent)."""
    if fast not in _ref:
        name = "libref_bench_fast.so" if fast else "libref_bench.so"
        path = os.path.join(ORACLE_DIR, "_ref", name)
        if not os.path.exists(path):
            _ref[fast] = None
        else:
            lib = ctypes.CDLL(path)
            lib.ref_bench_run.restype = ctypes.c_double
            lib.ref_bench_run.argtypes = _RUN_ARGS
            _ref[fast] = lib
    return _ref[fast]


def load_ref_api():
    """Direct handle on the reference library itself (public mbe_* symbols)."""
    path = os.path.join(ORACLE_DIR, "_ref", "libmberef.so")
    if not os.path.exists(path):
        return None
    return ctypes.CDLL(path)


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def run_cpu(fn, codec, soft, frames, seeds, n_threads=1, want_float=True, want_state=True):
    """Run a batch through `fn` (oracle mbo_run or reference ref_bench_run). frames: uint8
    [S][F][bits] (hard) or [S][F][bits][2] (soft: bit, reliability)."""
    frames = np.ascontiguousarray(frames, dtype=np.uint8)
    S, F = frames.shape[0], frames.shape[1]
    seeds = np.ascontiguousarray(seeds, dtype=np.uint32)
    out = dict(
        pcm=np.zeros((S, F, 160), np.int16),
        pcmf=np.zeros((S, F, 160), np.float32) if want_float else None,
        results=np.zeros((S, F, 6), np.int32),
        bits=np.zeros((S, F, PARAM_BITS[codec]), np.uint8),
        state=np.zeros((S, 3, PARMS_BYTES), np.uint8) if want_state else None,
    )
    out["seconds"] = fn(codec, int(bool(soft)), S, F, _ptr(frames), _ptr(seeds), _ptr(out["pcm"]),
                        _ptr(out["pcmf"]), _ptr(out["results"]), _ptr(out["bits"]), _ptr(out["state"]),
                        int(n_threads))
    return out


def random_hard_frames(codec, n_streams, n_frames, seed):
    rng = np.random.default_rng(seed)
    return rng.integers(0, 2, size=(n_streams, n_frames, FRAME_BITS[codec]), dtype=np.uint8)


def stream_seeds(n_streams, base=0xC0FFEE):
    return (np.arange(n_streams, dtype=np.uint64) + base).astype(np.uint32)


# ----------------------------------------------------------------------------------------------
# Channel encoders (inverse of the front-ends) so that tests can build VALID frames from chosen
# parameter bits: Golay/Hamming encode + PN scramble.  Pure numpy, per frame (small sizes only).
# ----------------------------------------------------------------------------------------------
_GOLAY_GEN = [0x63a, 0x31d, 0x7b4, 0x3da, 0x1ed, 0x6cc, 0x366, 0x1b3, 0x6e3, 0x54b, 0x49f, 0x475]
_HAM_ROWS = {0: [0x7f08, 0x78e4, 0x66d2, 0x55b1], 1: [0x7ac8, 0x3d64, 0x1eb2, 0x7591]}




def golay_encode(data12):
    ecc = 0
    for i in range(12):
        if (data12 >> (11 - i)) & 1:
            ecc ^= _GOLAY_GEN[i]
    return (data12 << 11) | ecc


def hamming_encode_hi11(data11, variant):
    """Codeword whose bits 14..4 equal data11 (MSB = bit 14) - the 11 bits the decoders extract."""
    rows = _HAM_ROWS[variant]
    base = data11 << 4
    for low in range(16):
        cw = base | low
        if all(bin(cw & r).count("1") % 2 == 0 for r in rows):
            return cw
    raise AssertionError("no codeword")


def pn_sequence(seed12, count):
    p = (16 * seed12) & 0xffff
    out = []
    for _ in range(count):
        p = (173 * p + 13849) & 0xffff
        out.append(p >> 15)
    return out


def encode_ambe_frame(bits49):
    """49 parameter bits -> valid char[4][24] AMBE 3600 frame (both AMBE codecs share the channel code)."""
    b = [int(x) for x in bits49]
    u0 = int("".join(map(str, b[0:12])), 2)
    u1 = int("".join(map(str, b[12:24])), 2)
    fr = np.zeros((4, 24), np.uint8)
    c0 = golay_encode(u0)
    for j in range(23):
        fr[0][j + 1] = (c0 >> j) & 1
    fr[0][0] = int(fr[0][1:].sum() & 1)  # overall even parity
    c1 = golay_encode(u1)
    pn = pn_sequence(u0, 23)
    k = 0
    for j in range(22, -1, -1):
        fr[1][j] = ((c1 >> j) & 1) ^ pn[k]
        k += 1
    for idx, j in enumerate(range(10, -1, -1)):
        fr[2][j] = b[24 + idx]
    for idx, j in enumerate(range(13, -1, -1)):
        fr[3][j] = b[35 + idx]
    return fr


def encode_imbe7200_frame(bits88):
    b = [int(x) for x in bits88]
    word = lambda lo, n: int("".join(map(str, b[lo:lo + n])), 2)
    fr = np.zeros((8, 23), np.uint8)
    u0 = word(0, 12)
    pn = pn_sequence(u0, 114)
    c0 = golay_encode(u0)
    for j in range(23):
        fr[0][j] = (c0 >> j) & 1
    k = 0
    for i in range(1, 4):
        cw = golay_encode(word(12 * i, 12))
        for j in range(22, -1, -1):
            fr[i][j] = ((cw >> j) & 1) ^ pn[k]
            k += 1
    for i in range(4, 7):
        cw = hamming_encode_hi11(word(48 + 11 * (i - 4), 11), 0)
        for j in range(14, -1, -1):
            fr[i][j] = ((cw >> j) & 1) ^ pn[k]
            k += 1
    for idx, j in enumerate(range(6, -1, -1)):
        fr[7][j] = b[81 + idx]
    return fr


def imbe7100_to_7200_layout(d88):
    """The K-dependent bit permutation between the IMBE 7100x4400 and 7200x4400 parameter layouts
    (what mbe_convertImbe7100to7200 does, /root/reference/src/imbe/imbe7100x4400.c:380-437)."""
    d = [int(x) for x in d88]
    b0 = int("".join(str(d[i]) for i in (1, 2, 3, 4, 5, 6, 86, 87)), 2)
    w0 = np.float32(np.float32(4 * np.pi) / np.float32(np.float32(b0) + 39.5))
    L = int(0.9254 * int((np.pi / float(w0)) + 0.25))
    K = int(np.float32(L + 2) / np.float32(3)) if L < 37 else 12
    out = [0] * 88
    out[87] = d[0]
    out[48 + K] = d[42]
    out[49 + K] = d[43]
    for i in range(K):
        out[48 + i] = d[44 + i]
    j, k = 0, 1
    while j < 87:
        out[j] = d[k]
        j += 1
        if j == 48:
            j += K + 2
        k += 1
        if k == 42:
            k += K + 2
    return np.array(out, np.uint8)


def encode_imbe7100_frame(d88):
    """88 data bits in the 7100x4400 LAYOUT (what mbe_eccImbe7100x4400Data emits, before the 7100 -> 7200 permutation)
    -> valid char[7][24] ProVoice frame: shortened Golay on C0 (7 data bits, five zero-extended), Golay on C1..C3, the
    7100 variant of Hamming(15,11) on C4 / C5, 23 raw bits, PN scrambling keyed by the 7 C0 data bits (the inverse of
    /root/reference/src/imbe/imbe7100x4400.c:99-122,152-212,291-334)."""
    b = [int(x) for x in d88]
    word = lambda lo, n: int("".join(map(str, b[lo:lo + n])), 2)
    fr = np.zeros((7, 24), np.uint8)
    u0 = word(0, 7)
    c0 = golay_encode(u0)                      # data bits 7..11 are zero, so code word bits 18..22 are zero
    for j in range(18):
        fr[0][j + 1] = (c0 >> j) & 1
    pn = pn_sequence(u0, 100)
    k = 0
    cw = golay_encode(word(7, 12))
    for j in range(23):
        fr[1][j + 1] = (cw >> j) & 1
    for j in range(23, -1, -1):                # the de-scrambler walks all 24 columns of row 1
        fr[1][j] ^= pn[k]
        k += 1
    for i in (2, 3):
        cw = golay_encode(word(19 + 12 * (i - 2), 12))
        for j in range(22, -1, -1):
            fr[i][j] = ((cw >> j) & 1) ^ pn[k]
            k += 1
    for i in (4, 5):
        cw = hamming_encode_hi11(word(43 + 11 * (i - 4), 11), 1)
        for j in range(14, -1, -1):
            fr[i][j] = ((cw >> j) & 1) ^ pn[k]
            k += 1
    for idx, j in enumerate(range(22, -1, -1)):
        fr[6][j] = b[65 + idx]
    return fr


def ecc_test_words(code, n, seed):
    """n soft-decision words for the block decoders (code 0 Golay(23,12), 1 / 2 Hamming(15,11) standard / 7100 layout):
    valid code words with 0..6 flipped bits (beyond what the hard decoders correct), reliabilities from five families that
    make cost ties and the "equals the hard decode" tie-break fire constantly: uniform 0..255, {0, 1, 2}, {k, k + 1},
    two-level {low, 255} with the flipped bits low, and two-level with the flipped bits claiming to be reliable.
    uint8 [n][len][2]."""
    rng = np.random.default_rng(seed)
    ln = 23 if code == 0 else 15
    if code == 0:
        cws = np.array([golay_encode(d) for d in range(4096)], np.uint32)
    else:
        cws = np.array([hamming_encode_hi11(d, code - 1) for d in range(2048)], np.uint32)
    cw = cws[rng.integers(0, len(cws), size=n)]
    bits = ((cw[:, None] >> np.arange(ln, dtype=np.uint32)) & 1).astype(np.uint8)
    nflip = rng.integers(0, 7, size=n)
    flip = (rng.random((n, ln)).argsort(axis=1).argsort(axis=1) < nflip[:, None])
    bits ^= flip.astype(np.uint8)
    fam = rng.integers(0, 5, size=n)
    k = rng.integers(0, 255, size=(n, 1))
    rel = np.where(fam[:, None] == 0, rng.integers(0, 256, size=(n, ln)),
          np.where(fam[:, None] == 1, rng.integers(0, 3, size=(n, ln)),
          np.where(fam[:, None] == 2, k + rng.integers(0, 2, size=(n, ln)),
          np.where(fam[:, None] == 3, np.where(flip, rng.integers(0, 64, size=(n, ln)), 255),
                   np.where(flip, 255, rng.integers(0, 64, size=(n, ln)))))))
    return np.ascontiguousarray(np.stack([bits, rel.astype(np.uint8)], axis=-1))


def oracle_ecc_blocks(code, words, soft, fast=True, n_threads=8):
    """oracle/mbe_oracle.c mbo_ecc_blocks: (decoded [n][len], status [n])."""
    o = load_oracle()
    n, ln = words.shape[0], words.shape[1]
    out = np.zeros((n, ln), np.uint8)
    st = np.zeros(n, np.int32)
    o.mbo_ecc_blocks(int(code), int(bool(soft)), int(bool(fast)), int(n), _ptr(np.ascontiguousarray(words)), _ptr(out), _ptr(st),
                     int(n_threads))
    return out, st


def mixed_frames(codec, S, F, seed):
    """random bits (repeats, mutes, re-initialisation), valid voice held for several frames (stable pitch: interpolated
    harmonics), valid frames with flipped bits, and for the AMBE codecs tone / erasure frames."""
    rng = np.random.default_rng(seed)
    fb = FRAME_BITS[codec]
    enc = {0: encode_imbe7200_frame, 1: encode_imbe7100_frame}.get(codec, encode_ambe_frame)
    frames = rng.integers(0, 2, size=(S, F, fb), dtype=np.uint8)
    for s in range(0, S, 2):
        f = 0
        while f < F:
            n = int(min(F - f, rng.integers(2, 9)))
            p = rng.integers(0, 2, size=PARAM_BITS[codec], dtype=np.uint8)
            if codec <= 1:
                p[codec] = 0
            elif rng.random() < 0.15:
                p[0:6] = 1                       # AMBE tone / erasure signatures
                if rng.random() < 0.5:
                    p[45:49] = 0
            fr = enc(p).reshape(-1)
            frames[s, f:f + n] = fr
            if rng.random() < 0.4:
                frames[s, f:f + n] ^= (rng.random((n, fb)) < 0.04).astype(np.uint8)
            f += n
    return frames


def oracle_rng_words(codec, soft, frames, seeds, n_threads=8):
    """Final RNG words [S][4] (export_rng layout) of each stream after the oracle decodes its frames from a fresh
    init_streams: the part of the end state that mbo_run does not return.  Replays the streams frame by frame
    (mbo_process_frame); ctypes releases the GIL, so threads over disjoint streams run in parallel."""
    from concurrent.futures import ThreadPoolExecutor
    o = load_oracle()
    frames = np.ascontiguousarray(frames, dtype=np.uint8)
    S, F = frames.shape[0], frames.shape[1]
    stride = frames[0, 0].nbytes
    out = np.zeros((S, 4), np.uint32)

    def work(lo_hi):
        bufs = dict(cur=np.zeros(PARMS_BYTES, np.uint8), prev=np.zeros(PARMS_BYTES, np.uint8),
                    enh=np.zeros(PARMS_BYTES, np.uint8), rng=np.zeros(16, np.uint8), pf=np.zeros(160, np.float32),
                    res=np.zeros(5, np.int32), d=np.zeros(88, np.uint8))
        p = {k: _ptr(v) for k, v in bufs.items()}
        for s in range(*lo_hi):
            o.mbo_rng_default(p["rng"])
            o.mbo_rng_seed(p["rng"], ctypes.c_uint32(int(seeds[s])))
            o.mbo_init_parms(p["cur"], p["prev"], p["enh"])
            for f in range(F):
                fr = ctypes.c_void_p(frames.ctypes.data + (s * F + f) * stride)
                o.mbo_process_frame(codec, int(bool(soft)), p["pf"], p["res"], fr, p["d"], p["cur"], p["prev"], p["enh"],
                                    p["rng"])
            out[s] = bufs["rng"].view(np.uint32)

    step = (S + n_threads - 1) // n_threads
    with ThreadPoolExecutor(n_threads) as ex:
        list(ex.map(work, [(lo, min(S, lo + step)) for lo in range(0, S, step)]))
    return out


# Tuning knobs of libmbe_b200 read from the environment once per process (knobs() in mbe_b200.cu); a test that varies
# them runs the library in a child process (tests/helpers/knob_child.py)
KNOBS = ("MBE_B200_PAD_SMEM", "MBE_B200_CHUNKS", "MBE_B200_TAPER", "MBE_B200_KSTREAMS", "MBE_B200_AUX", "MBE_B200_SPLIT",
         "MBE_B200_SKIP_KERNELS", "MBE_B200_DESC_MB")
KNOB_CHILD = os.path.join(ROOT, "tests", "helpers", "knob_child.py")


def run_knob_child(args, knobs, timeout):
    """Run tests/helpers/knob_child.py with `args` under exactly the knob settings `knobs` ({name: value}; every other
    knob is removed from the environment).  Returns its stdout; raises AssertionError with its output if it fails.  On a
    timeout subprocess.run kills the child, so nothing outlives the call."""
    env = {k: v for k, v in os.environ.items() if k not in KNOBS}
    env.update({k: str(v) for k, v in knobs.items()})
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [KNOB_CHILD] + [str(a) for a in args]
    p = subprocess.run(cmd, env=env, timeout=timeout, capture_output=True, text=True)
    if p.returncode != 0:
        raise AssertionError("knob child %s failed (%d) under %s:\n%s\n%s" % (args[0], p.returncode, knobs, p.stdout[-4000:],
                                                                            p.stderr[-4000:]))
    return p.stdout


def pipeline_plans(ns, knobs):
    """{n: mbe_b200_pipeline_plan(n)} under `knobs`, from a child process (no device needed)."""
    return {int(k): v for k, v in json.loads(run_knob_child(["plan"] + list(ns), knobs, timeout=120)).items()}


def soften(frames_hard, rng, flip_p=0.0, rel_ok=255, rel_bad_max=64):
    """Hard frames -> soft frames with seeded bit flips: unflipped bits get reliability `rel_ok`,
    flipped bits a reliability drawn from U[0, rel_bad_max)."""
    flips = rng.random(frames_hard.shape) < flip_p
    bits = frames_hard ^ flips.astype(np.uint8)
    rel = np.where(flips, rng.integers(0, rel_bad_max, size=frames_hard.shape), rel_ok).astype(np.uint8)
    return np.stack([bits, rel], axis=-1)


def fnv1a32(buf):
    h = 2166136261
    for x in bytes(buf):
        h ^= x
        h = (h * 16777619) & 0xffffffff
    return h


def parms_view(state_bytes):
    """Structured view of one 2604-byte mbe_parms blob."""
    raw = np.frombuffer(bytes(state_bytes), dtype=np.uint8)
    f = raw.view(np.float32)
    i = raw.view(np.int32)
    return dict(w0=f[0], L=i[1], K=i[2], Vl=i[3:60], Ml=f[60:117], log2Ml=f[117:174], PHIl=f[174:231],
                PSIl=f[231:288], gamma=f[288], tonePhase=raw.view(np.uint32)[289], swn=i[290], localEnergy=f[291],
                amplitudeThreshold=i[292], errorRate=f[293], errorCountTotal=i[294], errorCount4=i[295],
                repeatCount=i[296], mutingThreshold=f[297], previousUw=f[298:554], noiseSeed=f[554],
                noiseOverlap=f[555:651])
