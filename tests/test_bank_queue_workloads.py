"""The shaped workloads of tests/test_gpu_bank_queue.py reach the regimes they are built for, judged by the oracle's per-frame
work counts (mbo_run_work) and the bank kernel's grid-stride walk on a 148-SM B200 - without a GPU.

The bank kernel's frame queue (mbe_split_bank_kernel) has branches that only run when a warp fills its 32-frame window:
a window move with an open frame's sums in ws.carry, a frame ending exactly on a pass boundary, a window without any slot,
passes that mix the interpolated harmonics of several frames.  These tests make sure the workloads reach them, so that
the GPU comparison with the oracle checks what it is meant to check."""
import numpy as np
import pytest

import mbe_testlib as T

W_B200 = 148 * T.BANK_WARPS_PER_SM      # warps of the resident bank grid on a B200
DESC_BUDGET = 2048 << 20                # MBE_B200_DESC_MB's default: descriptors of one range


def _work(codec, mix):
    frames = T.shaped_frames(codec, mix)
    out = T.oracle_work(codec, 0, frames, T.stream_seeds(frames.shape[0]), want_float=False, want_state=False)
    return out["work"], out["results"]


def _queue(slots):
    """Per warp of the walk, the queue of padded slot counts: (walk [warp][visit], start and end of every visit's padded
    slots in its warp's queue).  Every pass takes the next 32 slots, so queue position p runs in pass p // 32 (a window
    move only skips positions after a frame without slots, which the mixes checked with this have none of)."""
    flat = slots.reshape(-1)
    walk = T.bank_walk(flat.size, W_B200)
    pad = np.where(walk >= 0, (flat[walk] + 3) & ~3, 0)
    end = np.cumsum(pad, axis=1)
    return walk, end - pad, end


@pytest.mark.parametrize("codec", T.SHAPED_CODECS)
@pytest.mark.parametrize("mix", T.SHAPED_MIXES)
def test_shaped_mix_reaches_its_regime(codec, mix):
    S, F = T.SHAPED_STREAMS, T.SHAPED_FRAMES
    # one range of the multi-kernel path under the default descriptor budget, at least 64 frames per bank warp
    assert S * F * T.DESC_BYTES <= DESC_BUDGET
    assert S * F >= 64 * W_B200
    work, results = _work(codec, mix)
    slots, k2, go = work[..., 0], work[..., 1], work[..., 2] == 1
    assert (results[..., 0] >= 0).all()
    assert ((slots == 0) | go).all() and (k2 <= slots).all() and slots.max() <= 112
    n_go = int(go.sum())
    if mix == "heavy":
        assert go.all()
        frac = ((slots >= 96) & (slots <= 112)).mean()
        assert frac >= 0.95, "%.3f of frames with 96-112 slots" % frac
    elif mix == "boundaries":
        pad = (slots + 3) & ~3
        for want in (32, 64, 96):
            assert (pad[go] == want).mean() >= 0.1, "padded count %d: %.3f" % (want, (pad[go] == want).mean())
        assert (slots[go] % 4 == 1).mean() >= 0.1
        assert (slots[go] > 0).all()
        _, start, end = _queue(slots)
        on_boundary = int(((end % 32 == 0) & (end > start)).sum())
        assert on_boundary >= S * F // 20, "%d frames end on a pass boundary" % on_boundary
    elif mix == "empty":
        zero_go = go & (slots == 0)
        assert zero_go.mean() >= 0.5 and (slots >= 96).mean() >= 0.05
        if codec == T.AMBE2450:
            assert ((results[..., 5] & T.FLAG_TONE) != 0).mean() >= 0.1
        walk, _, _ = _queue(slots)
        empty = np.where(walk >= 0, slots.reshape(-1)[walk] == 0, False)
        # 32 visits in a row without a slot, in warps that also run heavy frames
        run = np.cumsum(empty, axis=1)
        win32 = run[:, 32:] - run[:, :-32] == 32
        heavy = (np.where(walk >= 0, slots.reshape(-1)[walk], 0) >= 96).any(axis=1)
        warps = int((win32.any(axis=1) & heavy).sum())
        assert warps >= W_B200 // 2, "%d warps see heavy frames and an all-empty 32-frame window" % warps
    elif mix == "interp":
        assert go.all() and k2.sum() >= 6 * n_go
        walk, start, end = _queue(slots)
        k2w = np.where(walk >= 0, k2.reshape(-1)[walk], 0)
        # interpolated harmonics (l < 8) lead their frame's list: positions start .. start + k2 - 1
        has = k2w > 0
        first = start // 32
        last = (start + np.maximum(k2w, 1) - 1) // 32
        wi, vi = np.nonzero(has)
        owner = np.unique(np.concatenate([np.stack([wi, first[has], vi], 1), np.stack([wi, last[has], vi], 1)]), axis=0)
        _, cnt = np.unique(owner[:, :2], axis=0, return_counts=True)   # frames with interpolated slots per (warp, pass)
        mixed = int((cnt >= 2).sum())
        total_passes = int(np.ceil(end[:, -1] / 32).sum())
        assert mixed >= total_passes // 10, "%d of %d passes hold interpolated slots of two frames" % (mixed, total_passes)
    elif mix == "quiet":
        assert (slots == 0).all() and n_go > 0
