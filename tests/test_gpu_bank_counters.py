"""The bank kernel's pass counter (mbe_b200_kernel_timing counters[3], read through the C-ABI: Decoder.kernel_timing() keeps
to the first three).  The kernel streams the oscillator slots of the frames a warp visits through 32-slot passes across
frame boundaries (DESIGN 4.5), so on a launch with many frames per warp nearly every lane of every pass holds a slot; the
fused kernel counts nothing."""
import ctypes

import pytest
import torch

import mbe_testlib as T
from __graft_entry__ import load_package

pytestmark = pytest.mark.gpu


def counters(dec):
    ms = (ctypes.c_double * 3)()
    n = (ctypes.c_longlong * 3)()
    cnt = (ctypes.c_ulonglong * 4)()
    assert dec.lib.mbe_b200_kernel_timing(dec.h, ms, n, cnt) == 0
    return list(cnt)


def test_bank_passes_and_lane_fill():
    """IMBE 7200x4400 random bits, 4096 streams x 50 frames in one device-resident launch (~43 frames per warp of the
    resident bank grid): every slot runs in a pass (32 x passes >= slots), and the passes are at least 90 % full - frames
    padded to four slots and each warp's last pass are all that is left empty.  On the fused path all four counters stay 0."""
    pkg = load_package()
    codec, S, F = 0, 4096, 50
    dev = torch.device("cuda", 0)
    frames = torch.from_numpy(T.random_hard_frames(codec, S, F, 0xBA4C)).to(dev)
    pcm = torch.empty((S, F, 160), dtype=torch.int16, device=dev)
    res = torch.empty((S, F, 6), dtype=torch.int32, device=dev)
    dec = pkg.Decoder(max_streams=S, device=0)
    st = torch.cuda.Stream(dev)
    for path in (1, 0):
        dec.set_kernel_path(path)
        dec.init_streams(0, S, T.stream_seeds(S, 0xBA))
        dec.set_kernel_timing(True)
        dec.process_frames_dev(codec, 0, 0, S, F, frames.data_ptr(), pcm.data_ptr(), 0, res.data_ptr(), 0, st.cuda_stream)
        st.synchronize()
        slots, interp, synth, passes = counters(dec)
        dec.set_kernel_timing(False)
        if path == 1:
            assert 0 < synth <= S * F
            assert synth <= slots and interp <= slots
            assert 32 * passes >= slots > 0
            fill = slots / (32.0 * passes)
            assert fill >= 0.9, "lane fill %.4f (%d slots in %d passes)" % (fill, slots, passes)
        else:
            assert [slots, interp, synth, passes] == [0, 0, 0, 0]
    dec.close()
