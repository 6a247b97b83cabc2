"""GPU parity tests proper: the CUDA path (through the C-ABI, libmbe_b200.so) against the CPU oracle on the
same seeded inputs.  Bars against the oracle (check_batch and the long-stream test):
  - ECC error counts, result flags and decoded parameter bits: bit-exact;
  - int16 PCM and float PCM: bit-exact;
  - final mbe_parms triplets (previousUw / noiseOverlap / PHIl included): byte for byte.
Against the compiled reference (oracle/_ref, when present) - a build of the reference, not the oracle - int16 PCM keeps the
tolerance max |delta| <= 2 LSB with >= 99.99 % of samples exact; float PCM and state are reported."""
import numpy as np
import pytest

import mbe_testlib as T
from __graft_entry__ import load_package

pytestmark = pytest.mark.gpu

PCM_MAX_LSB = 2
PCM_EXACT_FRACTION = 0.9999


@pytest.fixture(scope="module")
def pkg():
    return load_package()


# every test that takes `dec` runs on both kernel paths of the frame entry points: the fused kernel and the parameter +
# synthesis kernel pair (mbe_b200_set_kernel_path, DESIGN 4.5); both must meet the same bars against the oracle
@pytest.fixture(scope="module", params=[0, 1], ids=["fused", "split"])
def dec(pkg, request):
    d = pkg.Decoder(max_streams=4096, device=0)
    d.set_kernel_path(request.param)
    assert d.kernel_path() == request.param
    yield d
    d.close()


def assert_pcm_exact(pcm, pcmf, want):
    """int16 and float PCM bit for bit against the oracle; the message locates the first difference."""
    for name, g, w in (("int16 PCM", pcm, want["pcm"]), ("float PCM", pcmf.view(np.uint32), want["pcmf"].view(np.uint32))):
        ne = g != w
        assert not ne.any(), "%s: %d of %d samples differ from the oracle, the first at (stream, frame, sample) %s" % (
            name, int(ne.sum()), ne.size, tuple(int(i) for i in np.argwhere(ne)[0]))


def assert_state_exact(st, want_state):
    """Final mbe_parms triplets byte for byte against the oracle; the message names the first differing field."""
    ne = st != want_state
    if ne.any():
        s, k, byte = (int(i) for i in np.argwhere(ne)[0])
        field = max((off, name) for name, off in T.OFF.items() if off <= byte)[1]
        raise AssertionError("final state differs from the oracle in %d streams, the first: stream %d, %s parms, field %s "
                             "(byte %d)" % (int(ne.any(axis=(1, 2)).sum()), s, ("cur", "prev", "enh")[k], field, byte))


def check_batch(dec, codec, soft, frames, seeds):
    S = frames.shape[0]
    dec.init_streams(0, S, seeds)
    got = dec.process_frames(codec, frames, soft=soft, want_float=True)
    want = T.run_cpu(T.load_oracle().mbo_run, codec, soft, frames, seeds, n_threads=8)
    res = got["results"]
    assert np.array_equal(res["status"], want["results"][..., 0])
    assert np.array_equal(got["bits"], want["bits"])
    assert np.array_equal(res["c0_errors"], want["results"][..., 1])
    assert np.array_equal(res["protected_errors"], want["results"][..., 2])
    assert np.array_equal(res["c4_errors"], want["results"][..., 3])
    assert np.array_equal(res["total_errors"], want["results"][..., 4])
    assert np.array_equal(res["flags"].astype(np.int64), want["results"][..., 5].astype(np.int64) & 0xffffffff)
    assert_pcm_exact(got["pcm"], got["pcmf"], want)
    st = dec.export_state(0, S)
    assert_state_exact(st, want["state"])
    out = dict(frames=int(res.size))
    # Second checker, one hop closer: the UNMODIFIED reference compiled by oracle/Makefile (Release flags, the parity
    # build of SURVEY 8(c)), when oracle/_ref travelled with the tree.  Bit-exact ECC and parameters, int16 PCM within the
    # tolerance of BASELINE.json: a build of the reference is not held to the oracle's bit-exact PCM bar.
    if T.ref_available(fast=False):
        ref = T.run_cpu(T.load_ref(fast=False).ref_bench_run, codec, soft, frames, seeds, n_threads=8)
        assert np.array_equal(res["status"], ref["results"][..., 0]), "status differs from the compiled reference"
        assert np.array_equal(got["bits"], ref["bits"]), "parameter bits differ from the compiled reference"
        for name, col in (("c0_errors", 1), ("protected_errors", 2), ("c4_errors", 3), ("total_errors", 4)):
            assert np.array_equal(res[name], ref["results"][..., col]), name + " differs from the compiled reference"
        assert np.array_equal(res["flags"].astype(np.int64), ref["results"][..., 5].astype(np.int64) & 0xffffffff)
        dr = np.abs(got["pcm"].astype(np.int32) - ref["pcm"].astype(np.int32))
        assert dr.max() <= PCM_MAX_LSB, "max |delta| vs the compiled reference = %d LSB" % dr.max()
        assert float((dr == 0).mean()) >= PCM_EXACT_FRACTION
        out["ref_exact"] = float((dr == 0).mean())
        out["ref_float_exact"] = float((got["pcmf"].view(np.uint32) == ref["pcmf"].view(np.uint32)).mean())
        out["ref_state_equal"] = bool(np.array_equal(st, ref["state"]))
    return out


@pytest.mark.parametrize("codec", [0, 1, 2, 3])
def test_random_hard_frames(dec, codec):
    frames = T.random_hard_frames(codec, 512, 50, 100 + codec)
    r = check_batch(dec, codec, 0, frames, T.stream_seeds(512))
    print(T.CODEC_NAMES[codec], r)


@pytest.mark.parametrize("codec", [0, 1, 2, 3])
def test_random_soft_frames(dec, codec):
    rng = np.random.default_rng(200 + codec)
    n = 16 if codec < 2 else 64
    bits = T.random_hard_frames(codec, n, 8, 210 + codec)
    rel = rng.integers(0, 256, size=bits.shape, dtype=np.uint8)
    r = check_batch(dec, codec, 1, np.stack([bits, rel], axis=-1), T.stream_seeds(n, 77))
    print(T.CODEC_NAMES[codec], r)


@pytest.mark.parametrize("codec,ber", [(3, 0.0), (3, 0.03), (2, 0.0), (2, 0.02), (0, 0.0), (0, 0.03), (1, 0.0), (1, 0.03)])
def test_encoded_voice_frames(dec, codec, ber):
    rng = np.random.default_rng(300 + codec + int(ber * 1000))
    S, F = 64, 50
    enc = {0: T.encode_imbe7200_frame, 1: T.encode_imbe7100_frame}.get(codec, T.encode_ambe_frame)
    frames = np.zeros((S, F, T.FRAME_BITS[codec]), np.uint8)
    for s in range(S):
        for f in range(F):
            p = rng.integers(0, 2, size=T.PARAM_BITS[codec], dtype=np.uint8)
            if codec <= 1:
                p[codec] = 0
            frames[s, f] = enc(p).reshape(-1)
    frames ^= (rng.random(frames.shape) < ber).astype(np.uint8)
    r = check_batch(dec, codec, 0, frames, T.stream_seeds(S, 5))
    print(T.CODEC_NAMES[codec], ber, r)


def test_ambe2400_tones_and_unvoiced(dec):
    rng = np.random.default_rng(4242)
    S, F = 96, 40
    frames = np.zeros((S, F, 96), np.uint8)
    for s in range(S):
        for f in range(F):
            p = rng.integers(0, 2, size=49, dtype=np.uint8)
            if (s + f // 5) % 3 == 0:
                p[0:6] = 1
            elif s % 2:
                p[38:42] = 1
            frames[s, f] = T.encode_ambe_frame(p).reshape(-1)
    r = check_batch(dec, T.AMBE2400, 0, frames, T.stream_seeds(S, 9))
    print(r)


def test_ambe2450_tone_frames(dec):
    rng = np.random.default_rng(777)
    S, F = 64, 24
    frames = np.zeros((S, F, 96), np.uint8)
    for s in range(S):
        for f in range(F):
            p = rng.integers(0, 2, size=49, dtype=np.uint8)
            if f % 4 == 1:
                p[0:6] = 1
                p[45:49] = 0
                tid = int(rng.integers(0, 200))
                p[12:20] = [(tid >> (7 - i)) & 1 for i in range(8)]
            frames[s, f] = T.encode_ambe_frame(p).reshape(-1)
    r = check_batch(dec, T.AMBE2450, 0, frames, T.stream_seeds(S, 3))
    print(r)


def test_soft_encoded_frames_with_flips(dec):
    rng = np.random.default_rng(555)
    for codec, S in ((0, 12), (3, 48)):
        F = 10
        enc = T.encode_imbe7200_frame if codec == 0 else T.encode_ambe_frame
        hard = np.zeros((S, F, T.FRAME_BITS[codec]), np.uint8)
        for s in range(S):
            for f in range(F):
                p = rng.integers(0, 2, size=T.PARAM_BITS[codec], dtype=np.uint8)
                p[0] = 0
                hard[s, f] = enc(p).reshape(-1)
        soft = T.soften(hard, rng, flip_p=0.10)
        r = check_batch(dec, codec, 1, soft, T.stream_seeds(S, 11))
        print(T.CODEC_NAMES[codec], r)


def test_invalid_bits_are_flagged_and_state_untouched(dec):
    frames = T.random_hard_frames(3, 8, 4, 31)
    frames[2, 1, 5] = 7            # not 0/1 -> MBE_STATUS_INVALID_BITS for that frame only
    seeds = T.stream_seeds(8)
    dec.init_streams(0, 8, seeds)
    got = dec.process_frames(3, frames, want_float=True)
    want = T.run_cpu(T.load_oracle().mbo_run, 3, 0, frames, seeds)
    assert got["results"]["status"][2, 1] == -2
    assert np.array_equal(got["results"]["status"], want["results"][..., 0])
    assert (got["pcm"][2, 1] == 0).all()
    d = np.abs(got["pcm"].astype(np.int32) - want["pcm"].astype(np.int32))
    assert d.max() <= PCM_MAX_LSB


def test_state_survives_split_launches(dec):
    """50 frames in one launch == 5 launches of 10 frames (state round-trips through HBM)."""
    frames = T.random_hard_frames(0, 64, 50, 909)
    seeds = T.stream_seeds(64)
    dec.init_streams(0, 64, seeds)
    a = dec.process_frames(0, frames)
    dec.init_streams(0, 64, seeds)
    parts = [dec.process_frames(0, frames[:, i:i + 10])["pcm"] for i in range(0, 50, 10)]
    assert np.array_equal(a["pcm"], np.concatenate(parts, axis=1))


def test_export_import_roundtrip(dec):
    frames = T.random_hard_frames(2, 32, 12, 77)
    seeds = T.stream_seeds(32)
    dec.init_streams(0, 32, seeds)
    dec.process_frames(2, frames[:, :6])
    st, rng = dec.export_state(0, 32), dec.export_rng(0, 32)
    a = dec.process_frames(2, frames[:, 6:])["pcm"]
    dec.import_state(st, 0)
    dec.import_rng(rng, 0)
    b = dec.process_frames(2, frames[:, 6:])["pcm"]
    assert np.array_equal(a, b)


def test_golden_pcm_fixture(dec):
    """tests/test_golden_pcm.c of the reference: one synthetic frame through mbe_synthesizeSpeechf +
    mbe_floattoshort; float hash 0x59741032 (scalar builds), int16 hash 0x4EDB8636."""
    o = T.load_oracle()
    cur = np.zeros((1, T.PARMS_BYTES), np.uint8)
    prev = np.zeros((1, T.PARMS_BYTES), np.uint8)
    enh = np.zeros((1, T.PARMS_BYTES), np.uint8)
    o.mbo_init_parms(T._ptr(cur), T._ptr(prev), T._ptr(enh))
    f, i = cur.view(np.float32).reshape(-1), cur.view(np.int32).reshape(-1)
    f[0] = np.float32(0.105)
    i[1] = 36
    for l in range(1, 37):
        i[3 + l] = 1 if l % 4 else 0
        f[60 + l] = np.float32(0.035) + np.float32(0.0015) * np.float32(l)
        f[174 + l] = np.float32(l) * np.float32(0.03)
        f[231 + l] = np.float32(l) * np.float32(0.02)
    prev[:] = cur
    # a batch of identical fixtures: every element must give the golden output
    n = 40
    curs, prevs = np.repeat(cur, n, axis=0).copy(), np.repeat(prev, n, axis=0).copy()
    pcmf, pcm = dec.synthesize_speech(curs, prevs, seeds=np.full(n, 0xC0FFEE, np.uint32))
    for k in (0, n - 1):
        assert T.fnv1a32(pcm[k].tobytes()) == 0x4EDB8636
        assert T.fnv1a32(pcmf[k].tobytes()) == 0x59741032
    assert (pcm == pcm[0]).all()


def test_floattoshort_edges(dec):
    """tests/test_floattoshort_parity.c: clip edges, NaN -> 0, +-Inf -> +-clip, truncation."""
    x = np.zeros(160, np.float32)
    edge = [0.0, -0.0, 1.0, -1.0, 4446.9, 4447.0, 4447.1, -4447.1, 1e9, -1e9, np.nan, np.inf, -np.inf, 0.14, -0.14,
            4681.0, -4681.0, 123.456, -123.456, 0.999 / 7]
    x[:len(edge)] = edge
    rng = np.random.default_rng(5)
    x[len(edge):] = rng.normal(0, 3000, 160 - len(edge)).astype(np.float32)
    got = dec.floattoshort(x)[0]
    want = np.zeros(160, np.int16)
    T.load_oracle().mbo_float_to_short(T._ptr(x), T._ptr(want))
    assert np.array_equal(got, want)


def test_staged_decode_then_data_equals_frame_path(dec):
    """mbe_decode*Frame followed by mbe_process*Data == mbe_process*Frame (README staged API)."""
    for codec in (0, 3):
        frames = T.random_hard_frames(codec, 48, 20, 1200 + codec)
        seeds = T.stream_seeds(48)
        dec.init_streams(0, 48, seeds)
        a = dec.process_frames(codec, frames)
        bits, res = dec.decode_frames(codec, frames)
        assert np.array_equal(bits.reshape(48, 20, -1), a["bits"])
        dec.init_streams(0, 48, seeds)
        b = dec.process_data(codec, bits.reshape(48, 20, -1), results=res.reshape(48, 20))
        assert np.array_equal(a["pcm"], b["pcm"])
        assert np.array_equal(a["results"]["flags"], b["results"]["flags"])


def test_process_data_without_context_uses_fallback_repeat_rules(dec):
    """result == NULL semantics (T4): no C0 context -> total-error fallback; with zero errors no repeats."""
    codec = 3
    frames = T.random_hard_frames(codec, 16, 10, 5150)
    bits, _ = dec.decode_frames(codec, frames)
    seeds = T.stream_seeds(16)
    dec.init_streams(0, 16, seeds)
    got = dec.process_data(codec, bits.reshape(16, 10, -1), results=None)
    o = T.load_oracle()
    # oracle: per stream, mbo_process_data with result = NULL
    import ctypes
    for s in range(16):
        cur = np.zeros(T.PARMS_BYTES, np.uint8); prev = cur.copy(); enh = cur.copy()
        rng = np.zeros(16, np.uint8)
        o.mbo_rng_default(T._ptr(rng)); o.mbo_rng_seed(T._ptr(rng), ctypes.c_uint32(int(seeds[s])))
        o.mbo_init_parms(T._ptr(cur), T._ptr(prev), T._ptr(enh))
        for f in range(10):
            out = np.zeros(160, np.float32); sh = np.zeros(160, np.int16)
            d = np.ascontiguousarray(bits.reshape(16, 10, -1)[s, f])
            o.mbo_process_data(codec, T._ptr(out), None, T._ptr(d), T._ptr(cur), T._ptr(prev), T._ptr(enh), T._ptr(rng))
            o.mbo_float_to_short(T._ptr(out), T._ptr(sh))
            assert np.abs(sh.astype(np.int32) - got["pcm"][s, f].astype(np.int32)).max() <= PCM_MAX_LSB


@pytest.mark.gpu
@pytest.mark.parametrize("codec", [0, 1, 2, 3])
def test_packed_frames_equal_unpacked(dec, pkg, codec):
    """SURVEY 8(f)-1: bit-packed channel frames give exactly what the one-byte-per-bit frames give (and the oracle)."""
    S, F = 96, 12
    frames = T.random_hard_frames(codec, S, F, 0x9ACC + codec)
    seeds = T.stream_seeds(S, 77)
    dec.init_streams(0, S, seeds)
    a = dec.process_frames(codec, frames, want_float=True)
    sa = dec.export_state(0, S)
    dec.init_streams(0, S, seeds)
    packed = pkg.pack_frames(codec, frames)
    assert packed.shape[-1] == pkg.packed_frame_bytes(codec) == dec.lib.mbe_b200_packed_frame_bytes(codec)
    b = dec.process_frames_packed(codec, packed, want_float=True)
    sb = dec.export_state(0, S)
    assert np.array_equal(a["pcm"], b["pcm"]) and np.array_equal(a["pcmf"].view(np.uint32), b["pcmf"].view(np.uint32))
    assert np.array_equal(a["bits"], b["bits"]) and np.array_equal(a["results"], b["results"])
    assert np.array_equal(sa, sb)
    want = T.run_cpu(T.load_oracle().mbo_run, codec, 0, frames, seeds, n_threads=8)
    assert np.array_equal(b["pcm"], want["pcm"]) and np.array_equal(b["bits"], want["bits"])


@pytest.mark.gpu
def test_normalized_float_output(dec):
    """SURVEY 8(f)-3: normalised float PCM = reference-scale float PCM x (7/32768), int16 PCM unchanged."""
    codec, S, F = 3, 64, 8
    frames = T.random_hard_frames(codec, S, F, 0x7F10)
    seeds = T.stream_seeds(S, 5)
    dec.init_streams(0, S, seeds)
    a = dec.process_frames(codec, frames, want_float=True)
    dec.init_streams(0, S, seeds)
    dec.set_normalized_float(True)
    try:
        b = dec.process_frames(codec, frames, want_float=True)
    finally:
        dec.set_normalized_float(False)
    assert np.array_equal(a["pcm"], b["pcm"])
    want = a["pcmf"] * np.float32(7.0 / 32768.0)
    assert np.array_equal(want.view(np.uint32), b["pcmf"].view(np.uint32))
    assert np.abs(b["pcmf"]).max() <= 0.951


@pytest.mark.gpu
def test_stream_window_and_degenerate_batches(dec):
    """first_stream / n_streams address a window of the state pool; empty batches are no-ops; one stream and one frame
    work (ragged blocks: 14 streams per block, so every size below exercises a partly filled block)."""
    codec = 0
    S, F = 37, 7
    frames = T.random_hard_frames(codec, S, F, 0xABCD)
    seeds = T.stream_seeds(S, 21)
    dec.init_streams(0, S, seeds)
    full = dec.process_frames(codec, frames)
    # the same streams living at an offset of the pool, processed in two windows and frame by frame
    off = 101
    dec.init_streams(off, S, seeds)
    a = dec.process_frames(codec, frames[:20], first_stream=off)
    b0 = dec.process_frames(codec, frames[20:, :3], first_stream=off + 20)
    b1 = dec.process_frames(codec, frames[20:, 3:4], first_stream=off + 20)
    b2 = dec.process_frames(codec, frames[20:, 4:], first_stream=off + 20)
    pcm = np.concatenate([a["pcm"], np.concatenate([b0["pcm"], b1["pcm"], b2["pcm"]], axis=1)], axis=0)
    assert np.array_equal(pcm, full["pcm"])
    assert np.array_equal(dec.export_state(0, S), dec.export_state(off, S))
    # degenerate sizes
    empty = dec.process_frames(codec, frames[:0])
    assert empty["pcm"].shape == (0, F, 160)
    none = dec.process_frames(codec, frames[:, :0])
    assert none["pcm"].shape == (S, 0, 160)
    dec.init_streams(0, 1, seeds[:1])
    one = dec.process_frames(codec, frames[:1, :1])
    assert np.array_equal(one["pcm"], full["pcm"][:1, :1])
    # out-of-range windows are refused, not clipped
    with pytest.raises(Exception):
        dec.process_frames(codec, frames, first_stream=dec.max_streams - 3)


@pytest.mark.parametrize("codec", [0, 1, 2, 3])
def test_soft_decode_degenerate_reliabilities(dec, codec):
    """Soft-decision ECC on reliability patterns that force ties and defeat the hard decode (the tie-break order of
    src/ecc/ecc.c:54-67,196-197 decides): all-equal reliabilities, erasures, two- and three-level reliabilities, flipped
    bits that claim to be reliable.  ECC stage only (mbe_b200_decode_frames) against the oracle, frame by frame."""
    import ctypes
    oracle = T.load_oracle()
    oracle.mbo_decode_frame.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    rng = np.random.default_rng(900 + codec)
    n = 40 if codec < 2 else 96
    fb, pb = T.FRAME_BITS[codec], T.PARAM_BITS[codec]
    enc = {0: T.encode_imbe7200_frame, 2: T.encode_ambe_frame, 3: T.encode_ambe_frame}.get(codec)
    patterns = {
        "all 0": lambda s: np.zeros(s, np.uint8),
        "all 255": lambda s: np.full(s, 255, np.uint8),
        "all 7": lambda s: np.full(s, 7, np.uint8),
        "0 or 255": lambda s: (rng.integers(0, 2, size=s) * 255).astype(np.uint8),
        "0..2": lambda s: rng.integers(0, 3, size=s).astype(np.uint8),
        "mostly 0, some 1": lambda s: (rng.random(s) < 0.2).astype(np.uint8),
    }
    for name, make in patterns.items():
        if enc is not None:
            hard = np.zeros((n, fb), np.uint8)
            for i in range(n):
                p = rng.integers(0, 2, size=pb, dtype=np.uint8)
                hard[i] = enc(p).reshape(-1)
            flips = rng.random(hard.shape) < 0.12
            bits_in = hard ^ flips.astype(np.uint8)
        else:
            bits_in = rng.integers(0, 2, size=(n, fb), dtype=np.uint8)
            flips = np.zeros(bits_in.shape, bool)
        rel = make(bits_in.shape)
        if name == "0 or 255":
            rel = np.where(flips, 255, rel).astype(np.uint8)  # the flipped bits claim to be reliable
        frames = np.ascontiguousarray(np.stack([bits_in, rel], axis=-1))
        got_bits, got_res = dec.decode_frames(codec, frames, soft=True)
        for i in range(n):
            wb = np.zeros(pb, np.uint8)
            wr = np.zeros(5, np.int32)
            rc = oracle.mbo_decode_frame(codec, 1, frames[i].ctypes.data, wb.ctypes.data, wr.ctypes.data)
            assert got_res["status"][i] == rc, (name, i)
            assert np.array_equal(got_bits[i], wb), (name, i)
            assert (got_res["c0_errors"][i], got_res["protected_errors"][i], got_res["c4_errors"][i],
                    got_res["total_errors"][i]) == tuple(int(x) for x in wr[:4]), (name, i)
            assert int(got_res["flags"][i]) == int(np.uint32(wr[4])), (name, i)


def _transmitted_positions(codec):
    """Frame positions (r*cols + c) that carry channel bits: everything for the random-bit tests except the unused
    corners of the reference's bit planes for the two 72/144-bit air interfaces."""
    if codec == 0:    # IMBE 7200x4400: 4 x 23 + 3 x 15 + 7 = 144 bits of char[8][23]
        pos = [r * 23 + c for r in range(4) for c in range(23)] + [r * 23 + c for r in range(4, 7) for c in range(15)]
        return pos + [7 * 23 + c for c in range(7)]
    if codec in (2, 3):  # AMBE 3600: 24 + 23 + 11 + 14 = 72 bits of char[4][24]
        return list(range(24)) + [24 + c for c in range(23)] + [48 + c for c in range(11)] + [72 + c for c in range(14)]
    return list(range(T.FRAME_BITS[codec]))


@pytest.mark.parametrize("codec", [0, 1, 2, 3])
def test_channel_map_deinterleaves_on_device(dec, pkg, codec):
    """SURVEY 8(f)-1: bit-packed frames in TRANSMISSION order + a caller-supplied interleave schedule
    (mbe_b200_set_channel_map) decode exactly like the same frames laid out as the reference's fr[rows][cols]."""
    rng = np.random.default_rng(0xC4A + codec)
    S, F = 64, 10
    pos = np.array(_transmitted_positions(codec), np.uint16)
    cmap = rng.permutation(pos)                       # transmitted bit k lands at frame position cmap[k]
    frames = T.random_hard_frames(codec, S, F, 0x77 + codec)
    mask = np.zeros(T.FRAME_BITS[codec], np.uint8)
    mask[pos] = 1
    frames &= mask                                    # positions the air interface does not carry are zero
    air = np.packbits(frames[..., cmap], axis=-1, bitorder="big")   # the caller's buffer: interleaved, eight bits per byte
    seeds = T.stream_seeds(S, 5)
    dec.init_streams(0, S, seeds)
    want = dec.process_frames(codec, frames, want_float=True)
    try:
        dec.set_channel_map(codec, cmap)
        assert dec.channel_frame_bytes(codec) == (len(cmap) + 7) // 8 == air.shape[-1]
        dec.init_streams(0, S, seeds)
        got = dec.process_frames_packed(codec, air, want_float=True)
        with pytest.raises(pkg.MbeB200Error):
            dec.set_channel_map(codec, np.array([0, 0], np.uint16))      # a position used twice
    finally:
        dec.set_channel_map(codec, None)
    assert dec.channel_frame_bytes(codec) == pkg.packed_frame_bytes(codec)
    for k in ("pcm", "bits", "results"):
        assert np.array_equal(got[k], want[k]), k
    assert np.array_equal(got["pcmf"].view(np.uint32), want["pcmf"].view(np.uint32))
    # the identity map is back: plain packed frames decode as before
    dec.init_streams(0, S, seeds)
    again = dec.process_frames_packed(codec, pkg.pack_frames(codec, frames))
    assert np.array_equal(again["pcm"], want["pcm"])


@pytest.mark.parametrize("F", [3, 33])
def test_host_pipeline_chunks_equal_single_launch(pkg, F):
    """The host-pointer call cuts a large batch into stream chunks (tapered at both ends, a ragged one in the middle) and
    pipelines copy-in / kernels / copy-out over several CUDA streams; every chunk must land where a single
    device-resident launch puts it (PCM, float PCM, results, bits, final state), for short and long launches."""
    import torch
    codec = 3
    S = 20000                                  # > 4 x 148 x 14 streams: several chunks, the last one ragged
    frames = np.ascontiguousarray(np.tile(T.random_hard_frames(codec, 250, F, 0xC0C), (S // 250, 1, 1)))
    seeds = T.stream_seeds(S, 0x99)
    d = pkg.Decoder(max_streams=S, device=0)
    d.init_streams(0, S, seeds)
    got = d.process_frames(codec, frames, want_float=True)
    st_host = d.export_state(0, S)
    d.init_streams(0, S, seeds)
    dev = torch.device("cuda", 0)
    d_fr = torch.from_numpy(frames).to(dev)
    d_pcm = torch.empty((S, F, 160), dtype=torch.int16, device=dev)
    d_pcmf = torch.empty((S, F, 160), dtype=torch.float32, device=dev)
    d_res = torch.empty((S, F, 6), dtype=torch.int32, device=dev)
    d_bits = torch.empty((S, F, pkg.PARAM_BITS[codec]), dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    d.process_frames_dev(codec, 0, 0, S, F, d_fr.data_ptr(), d_pcm.data_ptr(), d_pcmf.data_ptr(), d_res.data_ptr(), d_bits.data_ptr())
    d.synchronize()
    assert np.array_equal(got["pcm"], d_pcm.cpu().numpy())
    assert np.array_equal(got["pcmf"].view(np.uint32), d_pcmf.cpu().numpy().view(np.uint32))
    assert np.array_equal(got["bits"], d_bits.cpu().numpy())
    assert np.array_equal(got["results"].view(np.int32).reshape(S, F, 6), d_res.cpu().numpy())
    assert np.array_equal(st_host, d.export_state(0, S))
    d.close()


def test_short_launches_over_many_streams(pkg):
    """One or two frames per launch over many streams (what a real-time server does): 66 000 streams = 4715 blocks with a
    ragged last one, launches of 1, 2, 1, 2 frames; replicas of 300 distinct streams must equal the oracle wherever they
    sit in the grid, frame after frame, and so must the final state."""
    import torch
    codec, S, B, F = 3, 66000, 300, 6
    base = T.random_hard_frames(codec, B, F, 0x4E5)
    frames = np.ascontiguousarray(np.tile(base, ((S + B - 1) // B, 1, 1))[:S])
    seeds = np.tile(T.stream_seeds(B, 0x77), (S + B - 1) // B)[:S].astype(np.uint32)
    want = T.run_cpu(T.load_oracle().mbo_run, codec, 0, base, T.stream_seeds(B, 0x77), n_threads=8)
    dev = torch.device("cuda", 0)
    d_fr = torch.from_numpy(frames).to(dev)
    d = pkg.Decoder(max_streams=S, device=0)
    d.init_streams(0, S, seeds)
    d_pcm = torch.empty((S, F, 160), dtype=torch.int16, device=dev)
    d_res = torch.empty((S, F, 6), dtype=torch.int32, device=dev)
    for f0, nf in ((0, 1), (1, 2), (3, 1), (4, 2)):
        fr = d_fr[:, f0:f0 + nf].contiguous()
        pcm = torch.empty((S, nf, 160), dtype=torch.int16, device=dev)
        res = torch.empty((S, nf, 6), dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        d.process_frames_dev(codec, 0, 0, S, nf, fr.data_ptr(), pcm.data_ptr(), 0, res.data_ptr(), 0)
        d.synchronize()
        d_pcm[:, f0:f0 + nf] = pcm
        d_res[:, f0:f0 + nf] = res
    pcm, res, st = d_pcm.cpu().numpy(), d_res.cpu().numpy(), d.export_state(0, S)
    d.close()
    for k in (0, (S // B // 2) * B, (S // B - 1) * B):           # replicas at the start, the middle and the end of the grid
        assert np.array_equal(pcm[k:k + B], want["pcm"]), k
        assert np.array_equal(res[k:k + B, :, 4], want["results"][..., 4]), k
        assert np.array_equal(st[k:k + B], want["state"]), k


@pytest.mark.parametrize("codec", [0, 1, 2, 3])
def test_long_streams_stay_exact(dec, codec):
    """24 s of channel per stream (1200 frames x 48 streams), decoded in launches of 1 to 300 frames, against the oracle run
    in one go: steady voice (the same parameters held for several frames, so the pitch is stable and the low harmonics go
    through the phase-interpolated path), clean and noisy valid frames, random-bit bursts long enough to repeat, mute and
    re-initialise, then recovery.  Nothing may drift: parameter bits, results, int16 and float PCM exact over the whole
    run, final state byte for byte."""
    rng = np.random.default_rng(0x10C0 + codec)
    S, F, P = 48, 1200, 160
    fb = T.FRAME_BITS[codec]
    enc = {0: T.encode_imbe7200_frame, 1: T.encode_imbe7100_frame}.get(codec, T.encode_ambe_frame)
    pool = np.zeros((P, fb), np.uint8)
    for i in range(P):
        p = rng.integers(0, 2, size=T.PARAM_BITS[codec], dtype=np.uint8)
        if codec <= 1:
            p[codec] = 0        # most significant bit of b0 (bit 0 in the 7200 layout, bit 1 in the 7100 layout)
        pool[i] = enc(p).reshape(-1)
    frames = np.zeros((S, F, fb), np.uint8)
    for s in range(S):
        f = 0
        while f < F:
            kind = rng.integers(0, 4)
            n = int(min(F - f, rng.integers(3, 40)))
            if kind == 0:        # steady voice: one frame held
                frames[s, f:f + n] = pool[rng.integers(0, P)]
            elif kind == 1:      # changing clean voice
                frames[s, f:f + n] = pool[rng.integers(0, P, size=n)]
            elif kind == 2:      # noisy voice, 3 % flipped bits
                frames[s, f:f + n] = pool[rng.integers(0, P, size=n)] ^ (rng.random((n, fb)) < 0.03).astype(np.uint8)
            else:                # lost channel
                n = min(n, 14)
                frames[s, f:f + n] = rng.integers(0, 2, size=(n, fb), dtype=np.uint8)
            f += n
    seeds = T.stream_seeds(S, 0x10C)
    want = T.run_cpu(T.load_oracle().mbo_run, codec, 0, frames, seeds, n_threads=8)
    dec.init_streams(0, S, seeds)
    cuts, f = [], 0
    for n in [1, 1, 2, 7, 50, 139, 300, 1, 3, 200, 96, 400]:
        cuts.append((f, min(F, f + n)))
        f = min(F, f + n)
    assert f == F
    parts = [dec.process_frames(codec, np.ascontiguousarray(frames[:, a:b]), want_float=True) for a, b in cuts if b > a]
    pcm = np.concatenate([p["pcm"] for p in parts], axis=1)
    pcmf = np.concatenate([p["pcmf"] for p in parts], axis=1)
    bits = np.concatenate([p["bits"] for p in parts], axis=1)
    res = np.concatenate([p["results"] for p in parts], axis=1)
    assert np.array_equal(bits, want["bits"])
    assert np.array_equal(res["status"], want["results"][..., 0])
    assert np.array_equal(res["total_errors"], want["results"][..., 4])
    assert np.array_equal(res["flags"].astype(np.int64), want["results"][..., 5].astype(np.int64) & 0xffffffff)
    assert_pcm_exact(pcm, pcmf, want)
    assert_state_exact(dec.export_state(0, S), want["state"])
