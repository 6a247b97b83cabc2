"""Indexed batches (mbe_b200_process_indexed*, *_indexed state calls, pool forms): element i of a call decodes stream slot
slots[i], any set of slots in any order.  Outputs must equal the CPU oracle run over each slot's own frame history
(float PCM bitwise, int16 PCM, results, parameter bits, final mbe_parms triplets and RNG words byte for byte), slots no
call lists must not move, and a slot list with an out-of-range or repeated slot is rejected element by element (frame
calls) or as a whole (state calls)."""
import ctypes

import numpy as np
import pytest

import mbe_testlib as T
from __graft_entry__ import load_package

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg():
    return load_package()


# both kernel paths of the frame entry points: the fused kernel and the parameter + synthesis kernels
@pytest.fixture(params=[0, 1], ids=["fused", "split"])
def path(request):
    return request.param


def _decoder(pkg, max_streams, path):
    d = pkg.Decoder(max_streams=max_streams, device=0)
    d.set_kernel_path(path)
    return d


class OracleStream:
    """One stream of the CPU oracle, frame by frame (mbo_process_frame), state and RNG carried between calls."""

    def __init__(self, seed):
        self.o = T.load_oracle()
        self.cur, self.prev, self.enh = (np.zeros(T.PARMS_BYTES, np.uint8) for _ in range(3))
        self.rng = np.zeros(16, np.uint8)
        self.o.mbo_rng_default(T._ptr(self.rng))
        self.o.mbo_rng_seed(T._ptr(self.rng), ctypes.c_uint32(int(seed)))
        self.o.mbo_init_parms(T._ptr(self.cur), T._ptr(self.prev), T._ptr(self.enh))

    def run(self, codec, soft, frames):
        F = frames.shape[0]
        out = dict(pcm=np.zeros((F, 160), np.int16), pcmf=np.zeros((F, 160), np.float32),
                   results=np.zeros((F, 6), np.int32), bits=np.zeros((F, T.PARAM_BITS[codec]), np.uint8))
        for f in range(F):
            fr = np.ascontiguousarray(frames[f])
            pf = np.zeros(160, np.float32)
            res = np.zeros(5, np.int32)   # mbo_result: c0, protected, c4, total errors, flags
            d = np.zeros(88, np.uint8)
            ret = self.o.mbo_process_frame(codec, int(soft), T._ptr(pf), T._ptr(res), T._ptr(fr), T._ptr(d),
                                           T._ptr(self.cur), T._ptr(self.prev), T._ptr(self.enh), T._ptr(self.rng))
            if ret >= 0:
                out["pcmf"][f] = pf
                self.o.mbo_float_to_short(T._ptr(pf), T._ptr(out["pcm"][f]))
            out["results"][f, 0] = ret
            out["results"][f, 1:] = res
            out["bits"][f] = d[:T.PARAM_BITS[codec]]
        return out

    def state(self):
        return np.stack([self.cur, self.prev, self.enh])

    def rng_words(self):
        return self.rng.view(np.uint32).copy()


def _assert_element(got, i, want):
    assert np.array_equal(got["pcm"][i], want["pcm"]), i
    assert np.array_equal(got["pcmf"][i].view(np.uint32), want["pcmf"].view(np.uint32)), i
    assert np.array_equal(got["results"][i].view(np.int32).reshape(-1, 6), want["results"]), i
    assert np.array_equal(got["bits"][i], want["bits"]), i


def _assert_rejected(got, i):
    r = got["results"][i]
    assert np.all(r["status"] == -1), i
    for k in ("c0_errors", "protected_errors", "c4_errors", "total_errors", "flags"):
        assert np.all(r[k] == 0), (i, k)
    assert not got["pcm"][i].any() and not got["pcmf"][i].view(np.uint32).any() and not got["bits"][i].any(), i


def _frames(codec, input, n, F, rng, cmap=None):
    """(channel frames for the library, the same frames as the oracle reads them)"""
    hard = rng.integers(0, 2, size=(n, F, T.FRAME_BITS[codec]), dtype=np.uint8)
    if input == 1:
        soft = T.soften(hard, rng, flip_p=0.05)
        return soft, soft
    if input == 2:
        return np.packbits(hard[..., cmap], axis=-1, bitorder="big"), hard
    return hard, hard


CASES = [(c, i) for c in range(4) for i in (0, 1)] + [(0, 2)]


@pytest.mark.parametrize("codec,input", CASES, ids=["c%d-%s" % (c, ("hard", "soft", "packed")[i]) for c, i in CASES])
def test_scattered_slots_across_calls(pkg, path, codec, input):
    M = 300
    rng = np.random.default_rng(0x1D0 + 7 * codec + input)
    d = _decoder(pkg, M, path)
    cmap = None
    if input == 2:   # a non-identity channel map: transmitted bit k lands at frame position cmap[k]
        cmap = rng.permutation(T.FRAME_BITS[codec]).astype(np.uint16)
        d.set_channel_map(codec, cmap)
    seeds = T.stream_seeds(M, 0x5107)
    order = rng.permutation(M).astype(np.int32)
    d.init_streams_indexed(order, seeds[order])
    before = d.export_state(0, M)
    rng_before = d.export_rng(0, M)

    A = rng.permutation(M)[:120].astype(np.int32)                           # unsorted
    notA = np.setdiff1d(np.arange(M), A)
    B = rng.permutation(np.concatenate([A[:50], rng.choice(notA, 70, replace=False)])).astype(np.int32)
    FA, FB = 5, 3
    inA, orA = _frames(codec, input, A.size, FA, rng, cmap)
    inB, orB = _frames(codec, input, B.size, FB, rng, cmap)
    got_a = d.process_indexed(codec, A, inA, input=input, want_float=True)
    got_b = d.process_indexed(codec, B, inB, input=input, want_float=True)

    soft = input == 1
    streams = {}
    for i, s in enumerate(A):
        streams[int(s)] = OracleStream(seeds[s])
        _assert_element(got_a, i, streams[int(s)].run(codec, soft, orA[i]))
    for i, s in enumerate(B):
        if int(s) not in streams:
            streams[int(s)] = OracleStream(seeds[s])
        _assert_element(got_b, i, streams[int(s)].run(codec, soft, orB[i]))

    both = np.array(sorted(streams), np.int32)
    st = d.export_state_indexed(both)
    rw = d.export_rng_indexed(both)
    for k, s in enumerate(both):
        assert np.array_equal(st[k], streams[int(s)].state()), s
        assert np.array_equal(rw[k], streams[int(s)].rng_words()), s
    idle = np.setdiff1d(np.arange(M), both)
    assert idle.size > 0
    assert np.array_equal(d.export_state(0, M)[idle], before[idle])
    assert np.array_equal(d.export_rng(0, M)[idle], rng_before[idle])
    if input == 2:
        d.set_channel_map(codec, None)
    d.close()


def test_identity_list_equals_contiguous(pkg, path):
    """slots = [f, f + n) gives exactly what process_frames gives on that range, across several pipeline chunks and
    several descriptor ranges of the multi-kernel path."""
    codec, S, F, f0 = 3, 20000, 3, 37
    frames = np.ascontiguousarray(np.tile(T.random_hard_frames(codec, 250, F, 0x1DE), (S // 250, 1, 1)))
    seeds = T.stream_seeds(S + f0 + 11, 0x33)
    d = _decoder(pkg, S + f0 + 11, path)
    d.init_streams(0, None, seeds)
    want = d.process_frames(codec, frames, first_stream=f0, want_float=True)
    want_state, want_rng = d.export_state(0, None), d.export_rng(0, None)
    d.init_streams(0, None, seeds)
    got = d.process_indexed(codec, np.arange(f0, f0 + S, dtype=np.int32), frames, want_float=True)
    for k in ("pcm", "bits", "results"):
        assert np.array_equal(got[k], want[k]), k
    assert np.array_equal(got["pcmf"].view(np.uint32), want["pcmf"].view(np.uint32))
    assert np.array_equal(d.export_state(0, None), want_state)
    assert np.array_equal(d.export_rng(0, None), want_rng)
    d.close()


def _rejection_case(M):
    """identity list over M slots with element 5 -> -1, element 100 -> M, and the last element repeating element 3's slot
    (the last pipeline chunk, far from the first occurrence); the rejected elements are also the slots no element owns"""
    slots = np.arange(M, dtype=np.int32)
    slots[5], slots[100], slots[M - 1] = -1, M, 3
    return slots, (5, 100, M - 1)


def test_rejection_host_and_dev(pkg, path):
    import torch
    codec, M, F, B = 3, 20000, 2, 250
    base = T.random_hard_frames(codec, B, F, 0x2E1)
    base_seeds = T.stream_seeds(B, 0x71)
    frames = np.ascontiguousarray(np.tile(base, (M // B, 1, 1)))
    seeds = np.tile(base_seeds, M // B).astype(np.uint32)
    want = T.run_cpu(T.load_oracle().mbo_run, codec, 0, base, base_seeds, n_threads=8)
    slots, rejected = _rejection_case(M)
    unowned = rejected
    assert M > 4 * 148 * 14    # more than one pipeline chunk
    d = _decoder(pkg, M, path)

    def check(got):
        for i in rejected:
            _assert_rejected(got, i)
        ok = np.setdiff1d(np.arange(M), rejected)
        k = ok % B
        assert np.array_equal(got["pcm"][ok], want["pcm"][k])
        assert np.array_equal(got["pcmf"][ok].view(np.uint32), want["pcmf"][k].view(np.uint32))
        assert np.array_equal(got["bits"][ok], want["bits"][k])
        assert np.array_equal(got["results"][ok].view(np.int32).reshape(-1, F, 6), want["results"][k])
        st = d.export_state(0, M)
        for s in unowned:
            assert np.array_equal(st[s], before[s]), s
        owned = np.setdiff1d(np.arange(M), unowned)
        assert np.array_equal(st[owned], want["state"][owned % B])

    # host call: pipeline chunks, the repeat in the last one
    d.init_streams(0, M, seeds)
    before = d.export_state(0, M)
    check(d.process_indexed(codec, slots, frames, want_float=True))

    # _dev on a caller's torch stream with a device slot list; outputs pre-filled with garbage
    d.init_streams(0, M, seeds)
    dev = torch.device("cuda", 0)
    d_slots = torch.from_numpy(slots).to(dev)
    d_fr = torch.from_numpy(frames).to(dev)
    d_pcm = torch.full((M, F, 160), 0x5555, dtype=torch.int16, device=dev)
    d_pcmf = torch.full((M, F, 160), 1.5, dtype=torch.float32, device=dev)
    d_res = torch.full((M, F, 6), 77, dtype=torch.int32, device=dev)
    d_bits = torch.full((M, F, T.PARAM_BITS[codec]), 9, dtype=torch.uint8, device=dev)
    s = torch.cuda.Stream(device=dev)
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        d.process_indexed_dev(codec, pkg.INPUT_HARD, d_slots.data_ptr(), M, F, d_fr.data_ptr(), d_pcm.data_ptr(),
                              d_pcmf.data_ptr(), d_res.data_ptr(), d_bits.data_ptr(), cuda_stream=s.cuda_stream)
    s.synchronize()
    got = dict(pcm=d_pcm.cpu().numpy(), pcmf=d_pcmf.cpu().numpy(), bits=d_bits.cpu().numpy(),
               results=d_res.cpu().numpy().view(pkg.RESULT_DTYPE).reshape(M, F))
    check(got)

    # state calls: the whole call fails, nothing moves
    st0, rng0 = d.export_state(0, M), d.export_rng(0, M)
    for bad in ([0, -1], [0, M], [1, 1]):
        bad = np.array(bad, np.int32)
        for call in (lambda: d.init_streams_indexed(bad, np.ones(2, np.uint32)),
                     lambda: d.export_state_indexed(bad),
                     lambda: d.import_state_indexed(bad, np.zeros((2, 3, T.PARMS_BYTES), np.uint8)),
                     lambda: d.export_rng_indexed(bad),
                     lambda: d.import_rng_indexed(bad, np.zeros((2, 4), np.uint32))):
            with pytest.raises(pkg.MbeB200Error) as e:
                call()
            assert "(-1)" in str(e.value)
    assert np.array_equal(d.export_state(0, M), st0) and np.array_equal(d.export_rng(0, M), rng0)
    # empty calls launch nothing
    n0 = d.launches
    d.process_indexed(codec, np.zeros(0, np.int32), np.zeros((0, F, T.FRAME_BITS[codec]), np.uint8))
    d.process_indexed(codec, slots[:4], np.zeros((4, 0, T.FRAME_BITS[codec]), np.uint8))
    d.init_streams_indexed(np.zeros(0, np.int32))
    assert d.launches == n0
    d.close()


def test_submit_indexed_equals_process_indexed(pkg, path):
    codec, M, F = 0, 500, 4
    rng = np.random.default_rng(0x5B)
    slots = rng.permutation(M)[:333].astype(np.int32)
    frames = rng.integers(0, 2, size=(slots.size, F, T.FRAME_BITS[codec]), dtype=np.uint8)
    seeds = T.stream_seeds(M, 0x11)
    d = _decoder(pkg, M, path)
    d.init_streams(0, M, seeds)
    want = d.process_indexed(codec, slots, frames, want_float=True)
    want_state = d.export_state(0, M)
    d.init_streams(0, M, seeds)
    out = dict(pcm=pkg.host_alloc((slots.size, F, 160), np.int16), pcmf=pkg.host_alloc((slots.size, F, 160), np.float32),
               results=pkg.host_alloc((slots.size, F), pkg.RESULT_DTYPE),
               bits=pkg.host_alloc((slots.size, F, T.PARAM_BITS[codec]), np.uint8))
    try:
        d.submit_indexed(codec, slots, frames, out)
        d.wait()
        for k in ("pcm", "bits", "results"):
            assert np.array_equal(out[k], want[k]), k
        assert np.array_equal(out["pcmf"].view(np.uint32), want["pcmf"].view(np.uint32))
    finally:
        for a in out.values():
            pkg.host_free(a)
    assert np.array_equal(d.export_state(0, M), want_state)
    d.close()


@pytest.mark.parametrize("M,n_shards", [(9, 8), (100, 3)])
def test_pool_indexed_equals_context(pkg, M, n_shards):
    import torch
    codec, F = 2, 5
    rng = np.random.default_rng(0x9001 + M)
    seeds = T.stream_seeds(M, 0x4242)
    order = rng.permutation(M).astype(np.int32)
    # arbitrary order across shards, a repeated slot and two out-of-range ones
    some = rng.permutation(M)[: max(2, 2 * M // 3)]
    slots = np.concatenate([some, [some[0], -3, M]]).astype(np.int32)
    rng.shuffle(slots)
    frames = rng.integers(0, 2, size=(slots.size, F, T.FRAME_BITS[codec]), dtype=np.uint8)

    one = pkg.Decoder(max_streams=M, device=0)
    one.init_streams_indexed(order, seeds[order])
    init_state = one.export_state(0, M)
    want = one.process_indexed(codec, slots, frames, want_float=True)
    want_state = one.export_state(0, M)
    one.close()

    pool = pkg.Pool(M, devices=[i % torch.cuda.device_count() for i in range(n_shards)])
    assert len(pool.shards()) == n_shards
    pool.init_streams_indexed(order, seeds[order])
    assert np.array_equal(pool.export_state(0, M), init_state)
    got = pool.process_indexed(codec, slots, frames, want_float=True)
    for k in ("pcm", "bits", "results"):
        assert np.array_equal(got[k], want[k]), k
    assert np.array_equal(got["pcmf"].view(np.uint32), want["pcmf"].view(np.uint32))
    assert np.array_equal(pool.export_state(0, M), want_state)
    for i in np.nonzero((slots < 0) | (slots >= M))[0]:
        _assert_rejected(got, i)
    with pytest.raises(pkg.MbeB200Error):
        pool.init_streams_indexed(np.array([0, 0], np.int32))
    pool.close()
