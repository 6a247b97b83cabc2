"""Parity at BASELINE.json's full batch sizes through size-independent properties.

A full-size batch cannot be pushed through the CPU oracle in a test, so it is built from 512 distinct
(stream seed, frame sequence) pairs replicated across the batch: every replica must give byte-identical int16 and float
PCM, results and parameter bits wherever it sits in the grid (block position, ragged tail, pipeline chunk), and the
512 distinct streams are checked against the oracle.  Device buffers via torch (plumbing only)."""
import numpy as np
import pytest

import mbe_testlib as T
from __graft_entry__ import load_package

pytestmark = pytest.mark.gpu

BASE = 512


def _run_fullsize(codec, n_streams, n_frames, seed, base_frames=None, soft=0):
    import torch
    pkg = load_package()
    dev = torch.device("cuda", 0)
    if base_frames is None:
        base_frames = T.random_hard_frames(codec, BASE, n_frames, seed)
    BASE_N = base_frames.shape[0]
    reps = n_streams // BASE_N
    assert reps * BASE_N == n_streams
    base_seeds = T.stream_seeds(BASE_N, 0xBEEF)
    want = T.run_cpu(T.load_oracle().mbo_run, codec, soft, base_frames, base_seeds, n_threads=8)
    dec = pkg.Decoder(max_streams=n_streams, device=0)
    try:
        dec.init_streams(0, n_streams, np.tile(base_seeds, reps))
        d_base = torch.from_numpy(base_frames.reshape(BASE_N, n_frames, -1)).to(dev)
        d_frames = d_base.unsqueeze(0).expand(reps, -1, -1, -1).reshape(n_streams, n_frames, -1).contiguous()
        d_pcm = torch.empty((n_streams, n_frames, 160), dtype=torch.int16, device=dev)
        d_pcmf = torch.empty((n_streams, n_frames, 160), dtype=torch.float32, device=dev)
        d_res = torch.empty((n_streams, n_frames, 6), dtype=torch.int32, device=dev)
        d_bits = torch.empty((n_streams, n_frames, pkg.PARAM_BITS[codec]), dtype=torch.uint8, device=dev)
        # cuda_stream = 0 selects the context's own NON-BLOCKING stream, which does not wait for torch's legacy
        # default stream: finish the replication copy before the launch
        torch.cuda.synchronize()
        dec.process_frames_dev(codec, soft, 0, n_streams, n_frames, d_frames.data_ptr(), d_pcm.data_ptr(), d_pcmf.data_ptr(),
                               d_res.data_ptr(), d_bits.data_ptr())
        torch.cuda.synchronize()
        # every replica equals replica 0
        # (float PCM bit for bit: rounding to int16 would hide last-bit differences in the bank kernel's sums)
        for name, t in (("pcm", d_pcm), ("pcmf", d_pcmf.view(torch.int32)), ("results", d_res), ("bits", d_bits)):
            v = t.view(reps, BASE_N, -1)
            bad = (v != v[0:1]).any(dim=2)          # [replica][base stream]
            if bool(bad.any()):
                where = bad.nonzero()[:8].cpu().numpy().tolist()
                raise AssertionError("replicas of the same stream differ across the batch: %s, %d of %d streams, first (replica, "
                                     "base stream): %s" % (name, int(bad.sum()), n_streams, where))
        # replica 0 (and the last, ragged-tail one) equal the oracle
        for r in (0, reps - 1):
            sl = slice(r * BASE_N, (r + 1) * BASE_N)
            assert np.array_equal(d_pcm[sl].cpu().numpy(), want["pcm"])
            assert np.array_equal(d_pcmf[sl].cpu().numpy().view(np.uint32), want["pcmf"].view(np.uint32))
            assert np.array_equal(d_bits[sl].cpu().numpy(), want["bits"])
            assert np.array_equal(d_res[sl, :, 4].cpu().numpy(), want["results"][..., 4])
        # final state of the last replica equals the first replica's, byte for byte
        a = dec.export_state(0, BASE_N)
        b = dec.export_state(n_streams - BASE_N, BASE_N)
        assert np.array_equal(a, b)
    finally:
        dec.close()


def test_config2_ambe2450_65536_streams_x_50_frames():
    """BASELINE.json configs[1]: AMBE+2 3600x2450, 65,536 streams x 50 frames on one B200."""
    _run_fullsize(3, 65536, 50, 0x2450)


def test_config3_imbe7200_1m_streams_x_50_frames():
    """BASELINE.json configs[2] at its single-GPU size: IMBE 7200x4400, 1,048,576 streams x 50 frames (about 71 GB of HBM with
    float PCM)."""
    _run_fullsize(0, 1048576, 50, 0x7200)


def test_config4_ambe2400_tones_and_unvoiced_262144_streams():
    """BASELINE.json configs[3]: AMBE 3600x2400 (D-STAR) built from parameter bits: tone frames and unvoiced-heavy voice
    frames, Golay-encoded and PN-scrambled into valid channel frames; 262,144 streams x 50 frames."""
    rng = np.random.default_rng(0x2400)
    F = 50
    frames = np.zeros((BASE, F, 96), np.uint8)
    for s in range(BASE):
        for f in range(F):
            p = rng.integers(0, 2, size=49, dtype=np.uint8)
            if (s + f // 5) % 3 == 0:
                p[0:6] = 1          # b0 = 126/127: tone / silence frames
            elif s % 2:
                p[38:42] = 0        # V/UV codebook entry 0: every band unvoiced (FFT / WOLA / noise generator path)
            frames[s, f] = T.encode_ambe_frame(p).reshape(-1)
    _run_fullsize(2, 262144, F, 0, base_frames=frames)


def test_config5_mixed_codec_soft_decision_10pct_errors():
    """BASELINE.json configs[4] at its per-GPU size (1M streams / 8 GPUs = 131,072, a third per codec): valid encoded
    frames for all three codecs (IMBE 7100 through tests/mbe_testlib.encode_imbe7100_frame) with every channel bit flipped
    with p = 0.10, reliability 255 for unflipped and U[0,64) for flipped bits, soft-decision ECC, 50 frames."""
    rng = np.random.default_rng(0x50F7)
    F, B = 50, 32
    per_codec = 43680  # 1365 x 32
    for codec in (0, 1, 3):
        enc = {0: T.encode_imbe7200_frame, 1: T.encode_imbe7100_frame, 3: T.encode_ambe_frame}[codec]
        hard = np.zeros((B, F, T.FRAME_BITS[codec]), np.uint8)
        for s in range(B):
            for f in range(F):
                p = rng.integers(0, 2, size=T.PARAM_BITS[codec], dtype=np.uint8)
                p[1 if codec == 1 else 0] = 0   # most significant bit of b0: a valid fundamental
                hard[s, f] = enc(p).reshape(-1)
        soft = T.soften(hard, rng, flip_p=0.10)
        _run_fullsize(codec, per_codec, F, 0, base_frames=soft, soft=1)
