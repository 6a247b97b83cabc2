"""The bank kernel's frame queue (mbe_split_bank_kernel, DESIGN 4.5) against the oracle, float PCM bit for bit, at sizes where
every bank warp walks at least 64 frames and so fills and moves its 32-frame window many times.

The shaped workloads (mbe_testlib.shaped_frames; tests/test_bank_queue_workloads.py checks on the CPU that each reaches its
regime) put the queue's rare branches on every warp: 100+-slot frames whose sums wait in ws.carry across passes and window
moves, frames ending exactly on a pass boundary, windows without any slot, passes mixing the interpolated harmonics of
frames with different w0 changes, and zero-slot frames whose descriptor still holds an earlier launch's samples.  Both
kernel paths are checked; on the multi-kernel path the bank kernel's counters must equal the oracle's per-frame work."""
import numpy as np
import pytest
import torch

import mbe_testlib as T
from __graft_entry__ import load_package

pytestmark = pytest.mark.gpu

PATHS = [0, 1]
_want = {}


@pytest.fixture(scope="module")
def pkg():
    return load_package()


def _oracle(codec, mix):
    if (codec, mix) not in _want:
        frames = T.shaped_frames(codec, mix)
        seeds = T.stream_seeds(frames.shape[0], 0xBA2C)
        _want[(codec, mix)] = (frames, seeds, T.oracle_work(codec, 0, frames, seeds, n_threads=16))
    return _want[(codec, mix)]


def _bank_warps():
    return torch.cuda.get_device_properties(0).multi_processor_count * T.BANK_WARPS_PER_SM


def _decode_dev(dec, codec, d_frames):
    """One device-resident call on all streams of d_frames ([S][F][bits] on cuda:0); outputs on the device."""
    S, F = d_frames.shape[0], d_frames.shape[1]
    dev = d_frames.device
    out = dict(pcm=torch.empty((S, F, 160), dtype=torch.int16, device=dev),
               pcmf=torch.empty((S, F, 160), dtype=torch.float32, device=dev),
               results=torch.empty((S, F, 6), dtype=torch.int32, device=dev),
               bits=torch.empty((S, F, T.PARAM_BITS[codec]), dtype=torch.uint8, device=dev))
    torch.cuda.synchronize()     # (the context's stream does not wait for torch's copies)
    dec.process_frames_dev(codec, 0, 0, S, F, d_frames.data_ptr(), out["pcm"].data_ptr(), out["pcmf"].data_ptr(),
                           out["results"].data_ptr(), out["bits"].data_ptr())
    torch.cuda.synchronize()
    return out


def _assert_equal_replicated(got, want, label):
    """Device outputs of `reps` replicas of the oracle's streams: every replica equals the oracle, bit for bit."""
    dev = got["pcm"].device
    S = want["pcm"].shape[0]
    for name in ("pcmf", "pcm", "results", "bits"):
        g = got[name]
        w = torch.from_numpy(np.ascontiguousarray(want[name])).to(dev)
        if name == "pcmf":
            g, w = g.view(torch.int32), w.view(torch.int32)
        ne = (g.view((-1, S) + tuple(g.shape[1:])) != w.unsqueeze(0)).any(-1)   # [replica][stream][frame]
        if bool(ne.any()):
            r, s, f = (int(i) for i in ne.nonzero()[0])
            raise AssertionError("%s: %s differs from the oracle in %d frames, the first: replica %d, stream %d, frame %d" % (
                label, name, int(ne.sum()), r, s, f))


def _assert_state(dec, want_state, reps, label):
    S = want_state.shape[0]
    for r in range(reps):
        st = dec.export_state(r * S, S)
        ne = st != want_state
        if ne.any():
            s, k, byte = (int(i) for i in np.argwhere(ne)[0])
            raise AssertionError("%s: final state of replica %d differs from the oracle, first at stream %d, %s parms byte %d" % (
                label, r, s, ("cur", "prev", "enh")[k], byte))


@pytest.mark.parametrize("mix", ["heavy", "boundaries", "empty", "interp"])
@pytest.mark.parametrize("codec", T.SHAPED_CODECS)
@pytest.mark.parametrize("path", PATHS, ids=["fused", "split"])
def test_shaped_mix_against_the_oracle(pkg, path, codec, mix):
    """One device-resident call of SHAPED_STREAMS x SHAPED_FRAMES: float and int16 PCM, results, parameter bits and the final
    mbe_parms triplets equal the oracle.  Multi-kernel path: one bank launch, at least 64 frames per bank warp, its slot,
    interpolated-harmonic and frame counters equal to the oracle's totals, and its passes full."""
    frames, seeds, want = _oracle(codec, mix)
    S, F = frames.shape[0], frames.shape[1]
    work = want["work"]
    dec = pkg.Decoder(max_streams=S, device=0)
    try:
        dec.set_kernel_path(path)
        dec.init_streams(0, S, seeds)
        d_frames = torch.from_numpy(frames).to("cuda:0")
        dec.set_kernel_timing(True)
        got = _decode_dev(dec, codec, d_frames)
        (slots, interp, synth, passes), launches = T.counters(dec)
        dec.set_kernel_timing(False)
        label = "%s %s %s" % (("fused", "split")[path], T.CODEC_NAMES[codec], mix)
        _assert_equal_replicated(got, want, label)
        _assert_state(dec, want["state"], 1, label)
        if path == 0:
            assert [slots, interp, synth, passes] == [0, 0, 0, 0]
            return
        assert launches[1] == 1, "%d bank launches" % launches[1]
        assert S * F >= 64 * _bank_warps(), "%.1f frames per bank warp" % (S * F / _bank_warps())
        assert slots == int(work[..., 0].sum())
        assert interp == int(work[..., 1].sum())
        assert synth == int(work[..., 2].sum())
        assert 32 * passes >= slots
        fill = slots / (32.0 * passes) if passes else 0.0
        print("%s: %.1f frames per warp, %.1f slots per synthesised frame, lane fill %.4f, %d interpolated slots" % (
            label, S * F / _bank_warps(), slots / max(synth, 1), fill, interp))
        if mix in ("heavy", "boundaries"):
            assert fill >= 0.9, "lane fill %.4f (%d slots in %d passes)" % (fill, slots, passes)
    finally:
        dec.close()


@pytest.mark.parametrize("codec", T.SHAPED_CODECS)
@pytest.mark.parametrize("path", PATHS, ids=["fused", "split"])
def test_zero_slot_frames_over_stale_descriptors(pkg, path, codec):
    """On one context, heavy launches and then launches of the same shape whose frames run no slot, twice over: every zero-slot
    synthesis frame must get zero voiced samples, never what its descriptor kept from the heavy launch.  The device-resident
    call of six replicas (36 000 streams) is cut into at least four ranges, one per internal stream's descriptor buffer; the
    host call pipelines its chunks over the compute streams' buffers."""
    reps = 6
    hv_frames, seeds, hv = _oracle(codec, "heavy")
    qt_frames, qseeds, qt = _oracle(codec, "quiet")
    assert np.array_equal(seeds, qseeds)
    S = hv_frames.shape[0]
    dec = pkg.Decoder(max_streams=reps * S, device=0)
    try:
        dec.set_kernel_path(path)
        all_seeds = np.tile(seeds, reps)
        d_hv = torch.from_numpy(hv_frames).to("cuda:0").repeat(reps, 1, 1)
        d_qt = torch.from_numpy(qt_frames).to("cuda:0").repeat(reps, 1, 1)
        for rnd in range(2):
            for name, d_frames, want in (("heavy", d_hv, hv), ("quiet", d_qt, qt)):
                label = "%s %s round %d %s (device, %d replicas)" % (("fused", "split")[path], T.CODEC_NAMES[codec], rnd, name,
                                                                     reps)
                dec.init_streams(0, reps * S, all_seeds)
                dec.set_kernel_timing(True)
                got = _decode_dev(dec, codec, d_frames)
                (slots, _, synth, _), launches = T.counters(dec)
                dec.set_kernel_timing(False)
                _assert_equal_replicated(got, want, label)
                _assert_state(dec, want["state"], reps, label)
                if path == 1:
                    assert launches[1] >= 4, "%s: %d bank launches" % (label, launches[1])
                    assert slots == reps * int(want["work"][..., 0].sum()) and synth == reps * int(want["work"][..., 2].sum())
                del got
            for name, frames, want in (("heavy", hv_frames, hv), ("quiet", qt_frames, qt)):
                dec.init_streams(0, S, seeds)
                got = dec.process_frames(codec, frames, want_float=True)
                label = "%s %s round %d %s (host)" % (("fused", "split")[path], T.CODEC_NAMES[codec], rnd, name)
                assert np.array_equal(got["pcmf"].view(np.uint32), want["pcmf"].view(np.uint32)), label
                assert np.array_equal(got["pcm"], want["pcm"]), label
                assert np.array_equal(got["results"].view(np.int32).reshape(want["results"].shape), want["results"]), label
                assert np.array_equal(got["bits"], want["bits"]), label
                _assert_state(dec, want["state"], 1, label)
    finally:
        dec.close()
