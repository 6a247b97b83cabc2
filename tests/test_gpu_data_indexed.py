"""Indexed parameter-bit batches (mbe_b200_process_data_indexed[_dev], submit_data_indexed, pool_process_data_indexed):
element i decodes stream slot slots[i] from parameter bits with mbe_process<Codec>Data semantics, one byte per bit or
packed eight per byte, with or without a decode context.  Every output is compared with the CPU oracle's mbo_process_data
replayed per slot in call order: int16 PCM and float PCM bitwise, results field by field, final mbe_parms triplets and RNG
words byte for byte.  A rejected element (slot out of range or repeated) returns the caller's result input with status -1,
zero PCM, and moves no state."""
import ctypes
import json
import os

import numpy as np
import pytest

import mbe_testlib as T
from __graft_entry__ import load_package

pytestmark = pytest.mark.gpu

CHILD = os.path.join(T.ROOT, "tests", "helpers", "data_knob_child.py")


@pytest.fixture(scope="module")
def pkg():
    return load_package()


@pytest.fixture(params=[0, 1], ids=["fused", "split"])
def path(request):
    return request.param


def _decoder(pkg, max_streams, path):
    d = pkg.Decoder(max_streams=max_streams, device=0)
    d.set_kernel_path(path)
    return d


class OracleStream:
    """One stream of the CPU oracle, parameter frame by parameter frame (mbo_process_data), state and RNG carried."""

    def __init__(self, seed):
        self.o = T.load_oracle()
        self.cur, self.prev, self.enh = (np.zeros(T.PARMS_BYTES, np.uint8) for _ in range(3))
        self.rng = np.zeros(16, np.uint8)
        self.o.mbo_rng_default(T._ptr(self.rng))
        self.o.mbo_rng_seed(T._ptr(self.rng), ctypes.c_uint32(int(seed)))
        self.o.mbo_init_parms(T._ptr(self.cur), T._ptr(self.prev), T._ptr(self.enh))

    def run(self, codec, bits, res_in):
        """bits uint8 [F][param bits]; res_in: RESULT_DTYPE [F] decode contexts or None.  The library's outputs: a negative
        status leaves the PCM zero and the result the caller's input with only the status replaced."""
        F = bits.shape[0]
        out = dict(pcm=np.zeros((F, 160), np.int16), pcmf=np.zeros((F, 160), np.float32),
                   results=None if res_in is None else np.zeros((F, 6), np.int32))
        for f in range(F):
            d = np.ascontiguousarray(bits[f])
            pf = np.zeros(160, np.float32)
            r = None if res_in is None else np.ascontiguousarray(res_in[f]).view(np.int32)[1:].copy()
            ret = self.o.mbo_process_data(codec, T._ptr(pf), T._ptr(r), T._ptr(d), T._ptr(self.cur), T._ptr(self.prev),
                                          T._ptr(self.enh), T._ptr(self.rng))
            if ret >= 0:
                out["pcmf"][f] = pf
                self.o.mbo_float_to_short(T._ptr(pf), T._ptr(out["pcm"][f]))
            if r is not None:
                out["results"][f, 0] = ret
                out["results"][f, 1:] = r
        return out

    def state(self):
        return np.stack([self.cur, self.prev, self.enh])

    def rng_words(self):
        return self.rng.view(np.uint32).copy()


def contexts(pkg, n, F, rng, invalid_p=0.05):
    """Decode contexts: C0 / C4 valid flags set and unset, soft-input flag, C0 / protected / C4 counts that drive the repeat
    and erasure rules (totals consistent with them), and a few invalid contexts (a flag outside the context and status
    flags), which give status -1 with the context echoed."""
    r = np.zeros((n, F), pkg.RESULT_DTYPE)
    c0 = rng.integers(0, 5, size=(n, F))
    prot = rng.integers(0, 10, size=(n, F))
    r["c0_errors"] = c0
    r["protected_errors"] = prot
    r["c4_errors"] = np.minimum(rng.integers(0, 4, size=(n, F)), c0 + prot)
    r["total_errors"] = np.where(rng.random((n, F)) < 0.5, 0, c0 + prot)
    r["flags"] = rng.choice([0, 1, 2, 4, 6, 7], size=(n, F))
    bad = rng.random((n, F)) < invalid_p
    r["flags"][bad] |= 0x100
    r["status"] = rng.integers(-5, 50, size=(n, F))    # an input status is ignored and always replaced
    return r


def random_bits(codec, n, F, rng):
    return rng.integers(0, 2, size=(n, F, T.PARAM_BITS[codec]), dtype=np.uint8)


def _res_i32(r):
    return np.ascontiguousarray(r).view(np.int32).reshape(r.shape[0], r.shape[1], 6)


def _assert_element(got, i, want, what=""):
    assert np.array_equal(got["pcm"][i], want["pcm"]), (what, i)
    assert np.array_equal(got["pcmf"][i].view(np.uint32), want["pcmf"].view(np.uint32)), (what, i)
    if want["results"] is None:
        assert got["results"] is None
    else:
        g = _res_i32(got["results"][i:i + 1])[0]
        for k, name in enumerate(pkg_fields()):
            assert np.array_equal(g[:, k], want["results"][:, k]), (what, i, name)


def pkg_fields():
    return ("status", "c0_errors", "protected_errors", "c4_errors", "total_errors", "flags")


def _assert_rejected(got, i, res_in):
    """status -1, every other field the caller's input, zero PCM"""
    if res_in is not None:
        r = got["results"][i]
        assert np.all(r["status"] == -1), i
        for k in pkg_fields()[1:]:
            assert np.array_equal(r[k], res_in[i][k]), (i, k)
    assert not got["pcm"][i].any() and not got["pcmf"][i].view(np.uint32).any(), i


def _inputs(pkg, codec, bits, packed):
    return pkg.pack_params(codec, bits) if packed else bits


CASES = [(c, ctx, pk) for c in range(4) for ctx in (False, True) for pk in (False, True)]


@pytest.mark.parametrize("codec,ctx,packed", CASES,
                         ids=["c%d-%s-%s" % (c, "ctx" if x else "noctx", "packed" if p else "bytes") for c, x, p in CASES])
def test_scattered_slot_sets(pkg, path, codec, ctx, packed):
    M = 300
    rng = np.random.default_rng(0xDA7A + 8 * codec + 2 * ctx + packed)
    d = _decoder(pkg, M, path)
    seeds = T.stream_seeds(M, 0x5D07)
    order = rng.permutation(M).astype(np.int32)
    d.init_streams_indexed(order, seeds[order])
    before, rng_before = d.export_state(0, M), d.export_rng(0, M)

    A = rng.permutation(M)[:120].astype(np.int32)
    notA = np.setdiff1d(np.arange(M), A)
    B = rng.permutation(np.concatenate([A[:50], rng.choice(notA, 70, replace=False)])).astype(np.int32)
    C = rng.permutation(np.concatenate([B[:40], A[60:90]])).astype(np.int32)
    streams = {}
    for S, F in ((A, 5), (B, 3), (C, 4)):
        bits = random_bits(codec, S.size, F, rng)
        res = contexts(pkg, S.size, F, rng) if ctx else None
        got = d.process_data_indexed(codec, S, _inputs(pkg, codec, bits, packed), results=res, packed=packed,
                                     want_float=True)
        for i, s in enumerate(S):
            st = streams.setdefault(int(s), OracleStream(seeds[s]))
            _assert_element(got, i, st.run(codec, bits[i], res[i] if ctx else None))

    both = np.array(sorted(streams), np.int32)
    st, rw = d.export_state_indexed(both), d.export_rng_indexed(both)
    for k, s in enumerate(both):
        assert np.array_equal(st[k], streams[int(s)].state()), s
        assert np.array_equal(rw[k], streams[int(s)].rng_words()), s
    idle = np.setdiff1d(np.arange(M), both)
    assert idle.size > 0
    assert np.array_equal(d.export_state(0, M)[idle], before[idle])
    assert np.array_equal(d.export_rng(0, M)[idle], rng_before[idle])
    d.close()


def test_identity_list_equals_contiguous(pkg, path):
    """slots = [f0, f0 + n) gives exactly what process_data gives on that range, host (across pipeline chunks) and _dev."""
    import torch
    codec, S, F, f0 = 0, 9000, 3, 37
    M = S + f0 + 11
    rng = np.random.default_rng(0x1DDA)
    bits = np.ascontiguousarray(np.tile(random_bits(codec, 250, F, rng), (S // 250, 1, 1)))
    res = contexts(pkg, S, F, rng)
    seeds = T.stream_seeds(M, 0x34)
    ident = np.arange(f0, f0 + S, dtype=np.int32)
    assert len(T.pipeline_plans([S], {})[S]) > 1
    d = _decoder(pkg, M, path)

    d.init_streams(0, None, seeds)
    want = d.process_data(codec, bits, results=res, first_stream=f0, want_float=True)
    want_state, want_rng = d.export_state(0, None), d.export_rng(0, None)
    d.init_streams(0, None, seeds)
    got = d.process_data_indexed(codec, ident, bits, results=res, want_float=True)
    for k in ("pcm", "results"):
        assert np.array_equal(got[k], want[k]), k
    assert np.array_equal(got["pcmf"].view(np.uint32), want["pcmf"].view(np.uint32))
    assert np.array_equal(d.export_state(0, None), want_state)
    assert np.array_equal(d.export_rng(0, None), want_rng)

    # _dev: contiguous process_data_dev against the identity list, each on a caller's stream
    dev = torch.device("cuda", 0)
    outs = []
    for indexed in (False, True):
        d.init_streams(0, None, seeds)
        x = torch.from_numpy(bits).to(dev)
        r = torch.from_numpy(_res_i32(res)).to(dev)
        o_pcm = torch.full((S, F, 160), 0x5555, dtype=torch.int16, device=dev)
        o_pcmf = torch.full((S, F, 160), 1.5, dtype=torch.float32, device=dev)
        sl = torch.from_numpy(ident).to(dev)
        s = torch.cuda.Stream(device=dev)
        torch.cuda.synchronize()
        with torch.cuda.stream(s):
            if indexed:
                d.process_data_indexed_dev(codec, False, sl.data_ptr(), S, F, x.data_ptr(), r.data_ptr(), o_pcm.data_ptr(),
                                           o_pcmf.data_ptr(), cuda_stream=s.cuda_stream)
            else:
                d._check(d.lib.mbe_b200_process_data_dev(d.h, codec, f0, S, F, ctypes.c_void_p(x.data_ptr()),
                                                         ctypes.c_void_p(r.data_ptr()), ctypes.c_void_p(o_pcm.data_ptr()),
                                                         ctypes.c_void_p(o_pcmf.data_ptr()), ctypes.c_void_p(s.cuda_stream)),
                         "process_data_dev")
        s.synchronize()
        outs.append((o_pcm.cpu().numpy(), o_pcmf.cpu().numpy().view(np.uint32), r.cpu().numpy(), d.export_state(0, None),
                     d.export_rng(0, None)))
    for a, b in zip(*outs):
        assert np.array_equal(a, b)
    assert np.array_equal(outs[0][0], want["pcm"]) and np.array_equal(outs[0][2], _res_i32(want["results"]))
    d.close()


@pytest.mark.parametrize("codec", [0, 1, 2, 3])
def test_packed_equals_unpacked_and_invalid_bytes(pkg, path, codec):
    """Packed input gives exactly what one byte per bit gives (pad bits ignored); a byte other than 0 / 1 in unpacked input
    gives status -2 with the state untouched, as the oracle does."""
    M, F = 200, 6
    rng = np.random.default_rng(0xBACC + codec)
    seeds = T.stream_seeds(M, 0x77)
    slots = rng.permutation(M)[:150].astype(np.int32)
    bits = random_bits(codec, slots.size, F, rng)
    res = contexts(pkg, slots.size, F, rng)
    packed = pkg.pack_params(codec, bits)
    pb = T.PARAM_BITS[codec]
    if pb % 8:
        packed[..., -1] |= np.uint8((1 << (8 - pb % 8)) - 1)     # set every pad bit: they must be ignored
    d = _decoder(pkg, M, path)
    d.init_streams(0, M, seeds)
    a = d.process_data_indexed(codec, slots, bits, results=res, want_float=True)
    sa, ra = d.export_state(0, M), d.export_rng(0, M)
    d.init_streams(0, M, seeds)
    b = d.process_data_indexed(codec, slots, packed, results=res, packed=True, want_float=True)
    for k in ("pcm", "results"):
        assert np.array_equal(a[k], b[k]), k
    assert np.array_equal(a["pcmf"].view(np.uint32), b["pcmf"].view(np.uint32))
    assert np.array_equal(d.export_state(0, M), sa) and np.array_equal(d.export_rng(0, M), ra)

    # non-binary bytes: every third element gets a 2 or 255 in some frames
    bad = bits.copy()
    hit = np.zeros((slots.size, F), bool)
    hit[::3, ::2] = True
    pos = rng.integers(0, pb, size=(slots.size, F))
    val = rng.choice([2, 255], size=(slots.size, F)).astype(np.uint8)
    for i, f in zip(*np.nonzero(hit)):
        bad[i, f, pos[i, f]] = val[i, f]
    d.init_streams(0, M, seeds)
    got = d.process_data_indexed(codec, slots, bad, results=res, want_float=True)
    assert np.all(got["results"]["status"][hit & (res["flags"] < 0x100)] == -2)
    for i, s in enumerate(slots):
        o = OracleStream(seeds[s])
        _assert_element(got, i, o.run(codec, bad[i], res[i]))
        st = d.export_state_indexed(np.array([s], np.int32))[0]
        assert np.array_equal(st, o.state()), s
    d.close()


@pytest.mark.parametrize("codec", [0, 1, 2, 3])
def test_staged_path_equals_process_indexed(pkg, path, codec):
    """decode_frames followed by process_data_indexed (the bits and ECC results as the decode context) equals
    process_indexed on the same hard frames: PCM, results, state and RNG."""
    M, F = 400, 7
    rng = np.random.default_rng(0x57A6 + codec)
    seeds = T.stream_seeds(M, 0x99)
    slots = rng.permutation(M)[:250].astype(np.int32)
    frames = T.mixed_frames(codec, slots.size, F, 0x57A0 + codec)
    d = _decoder(pkg, M, path)
    d.init_streams(0, M, seeds)
    want = d.process_indexed(codec, slots, frames, want_float=True)
    ws, wr = d.export_state(0, M), d.export_rng(0, M)
    d.init_streams(0, M, seeds)
    bits, res = d.decode_frames(codec, frames)
    got = d.process_data_indexed(codec, slots, bits.reshape(slots.size, F, -1), results=res.reshape(slots.size, F),
                                 want_float=True)
    for k in ("pcm", "results"):
        assert np.array_equal(got[k], want[k]), k
    assert np.array_equal(got["pcmf"].view(np.uint32), want["pcmf"].view(np.uint32))
    assert np.array_equal(d.export_state(0, M), ws) and np.array_equal(d.export_rng(0, M), wr)
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
    rng = np.random.default_rng(0x2E2)
    base = random_bits(codec, B, F, rng)
    base_res = contexts(pkg, B, F, rng)
    base_seeds = T.stream_seeds(B, 0x72)
    bits = np.ascontiguousarray(np.tile(base, (M // B, 1, 1)))
    res = np.ascontiguousarray(np.tile(base_res, (M // B, 1)))
    seeds = np.tile(base_seeds, M // B).astype(np.uint32)
    want, want_state = [], []
    for k in range(B):
        o = OracleStream(base_seeds[k])
        want.append(o.run(codec, base[k], base_res[k]))
        want_state.append(o.state())
    slots, rejected = _rejection_case(M)
    assert len(T.pipeline_plans([M], {})[M]) > 1     # the repeat falls in another pipeline chunk
    d = _decoder(pkg, M, path)

    def check(got):
        for i in rejected:
            _assert_rejected(got, i, res)
        for i in np.setdiff1d(np.arange(M), rejected)[::7]:
            _assert_element(got, i, want[i % B])
        ok = np.setdiff1d(np.arange(M), rejected)
        assert np.array_equal(got["pcm"][ok], np.stack([w["pcm"] for w in want])[ok % B])
        assert np.array_equal(_res_i32(got["results"][ok]), np.stack([w["results"] for w in want])[ok % B])
        st = d.export_state(0, M)
        for s in rejected:       # the rejected elements' slots are exactly the ones no element owns
            assert np.array_equal(st[s], before[s]), s
        assert np.array_equal(st[ok], np.stack(want_state)[ok % B])

    # host call: pipeline chunks, the repeat in the last one
    d.init_streams(0, M, seeds)
    before = d.export_state(0, M)
    check(d.process_data_indexed(codec, slots, bits, results=res, want_float=True))
    # no decode context: nothing to echo, zero PCM still
    d.init_streams(0, M, seeds)
    got = d.process_data_indexed(codec, slots, bits, want_float=True)
    assert got["results"] is None
    for i in rejected:
        _assert_rejected(got, i, None)

    # _dev on a caller's torch stream, packed input; PCM outputs pre-filled with garbage
    d.init_streams(0, M, seeds)
    dev = torch.device("cuda", 0)
    d_slots = torch.from_numpy(slots).to(dev)
    d_bits = torch.from_numpy(pkg.pack_params(codec, bits)).to(dev)
    d_res = torch.from_numpy(_res_i32(res)).to(dev)
    d_pcm = torch.full((M, F, 160), 0x5555, dtype=torch.int16, device=dev)
    d_pcmf = torch.full((M, F, 160), 1.5, dtype=torch.float32, device=dev)
    s = torch.cuda.Stream(device=dev)
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        d.process_data_indexed_dev(codec, True, d_slots.data_ptr(), M, F, d_bits.data_ptr(), d_res.data_ptr(),
                                   d_pcm.data_ptr(), d_pcmf.data_ptr(), cuda_stream=s.cuda_stream)
    s.synchronize()
    check(dict(pcm=d_pcm.cpu().numpy(), pcmf=d_pcmf.cpu().numpy(),
               results=d_res.cpu().numpy().view(pkg.RESULT_DTYPE).reshape(M, F)))

    # empty calls launch nothing
    n0 = d.launches
    d.process_data_indexed(codec, np.zeros(0, np.int32), np.zeros((0, F, T.PARAM_BITS[codec]), np.uint8))
    d.process_data_indexed(codec, slots[:4], np.zeros((4, 0, T.PARAM_BITS[codec]), np.uint8))
    d.process_data_indexed_dev(codec, False, d_slots.data_ptr(), 0, F, d_bits.data_ptr(), 0, d_pcm.data_ptr())
    assert d.launches == n0
    # packed is 0 or 1
    assert d.lib.mbe_b200_process_data_indexed(d.h, codec, 2, ctypes.c_void_p(slots.ctypes.data), 4, F,
                                               ctypes.c_void_p(bits.ctypes.data), None, None, None) == -1
    d.close()


def test_submit_equals_process(pkg, path):
    codec, M, F = 0, 500, 4
    rng = np.random.default_rng(0x5C)
    slots = rng.permutation(M)[:333].astype(np.int32)
    bits = pkg.pack_params(codec, random_bits(codec, slots.size, F, rng))
    res = contexts(pkg, slots.size, F, rng)
    seeds = T.stream_seeds(M, 0x12)
    d = _decoder(pkg, M, path)
    d.init_streams(0, M, seeds)
    want = d.process_data_indexed(codec, slots, bits, results=res, packed=True, want_float=True)
    want_state = d.export_state(0, M)
    d.init_streams(0, M, seeds)
    out = dict(pcm=pkg.host_alloc((slots.size, F, 160), np.int16), pcmf=pkg.host_alloc((slots.size, F, 160), np.float32),
               results=pkg.host_alloc((slots.size, F), pkg.RESULT_DTYPE))
    try:
        out["results"][:] = res
        d.submit_data_indexed(codec, slots, bits, out, packed=True)
        with pytest.raises(pkg.MbeB200Error) as e:       # one submission pending per context
            d.submit_data_indexed(codec, slots, bits, out, packed=True)
        assert "(-1)" in str(e.value)
        with pytest.raises(pkg.MbeB200Error):            # host calls refuse while it is pending
            d.process_data_indexed(codec, slots, bits, results=res, packed=True)
        d.wait()
        for k in ("pcm", "results"):
            assert np.array_equal(out[k], want[k]), k
        assert np.array_equal(out["pcmf"].view(np.uint32), want["pcmf"].view(np.uint32))
    finally:
        for a in out.values():
            pkg.host_free(a)
    assert np.array_equal(d.export_state(0, M), want_state)
    d.close()


@pytest.mark.parametrize("M,n_shards", [(9, 8), (100, 3)])
def test_pool_equals_context(pkg, M, n_shards):
    import torch
    codec, F = 2, 5
    rng = np.random.default_rng(0x9002 + M)
    seeds = T.stream_seeds(M, 0x4243)
    order = rng.permutation(M).astype(np.int32)
    some = rng.permutation(M)[: max(2, 2 * M // 3)]
    slots = np.concatenate([some, [some[0], -3, M]]).astype(np.int32)
    rng.shuffle(slots)
    bits = random_bits(codec, slots.size, F, rng)
    res = contexts(pkg, slots.size, F, rng)

    one = pkg.Decoder(max_streams=M, device=0)
    one.init_streams_indexed(order, seeds[order])
    want = one.process_data_indexed(codec, slots, bits, results=res, want_float=True)
    want_state = one.export_state(0, M)
    one.close()

    pool = pkg.Pool(M, devices=[i % torch.cuda.device_count() for i in range(n_shards)])
    assert len(pool.shards()) == n_shards
    pool.init_streams_indexed(order, seeds[order])
    got = pool.process_data_indexed(codec, slots, bits, results=res, want_float=True)
    for k in ("pcm", "results"):
        assert np.array_equal(got[k], want[k]), k
    assert np.array_equal(got["pcmf"].view(np.uint32), want["pcmf"].view(np.uint32))
    assert np.array_equal(pool.export_state(0, M), want_state)
    rejected = np.nonzero((slots < 0) | (slots >= M))[0]
    assert rejected.size == 2
    for i in rejected:
        _assert_rejected(got, i, res)
    # packed through the pool
    pool.init_streams_indexed(order, seeds[order])
    got_p = pool.process_data_indexed(codec, slots, pkg.pack_params(codec, bits), results=res, packed=True, want_float=True)
    for k in ("pcm", "results"):
        assert np.array_equal(got_p[k], want[k]), k
    pool.close()


# ---- tuning knobs: the host pipeline of the indexed data calls, in a child process per setting ----------------------
KM, KFIRST, KS = 12000, 37, 9000
KCUTS = [(0, 3), (3, 8)]
KSETTINGS = [
    ("default", {}),
    ("desc1", {"MBE_B200_DESC_MB": 1}),
    ("chunks5-taper1", {"MBE_B200_CHUNKS": 5, "MBE_B200_TAPER": 1}),
    ("fused-chunks64-taper0", {"MBE_B200_SPLIT": 0, "MBE_B200_CHUNKS": 64, "MBE_B200_TAPER": 0}),
]


def _oracle_decode(codec, frames):
    """parameter bits and ECC results (the decode context) of hard frames, by the oracle (mbo_decode_frame)"""
    o = T.load_oracle()
    S, F = frames.shape[0], frames.shape[1]
    bits = np.zeros((S, F, T.PARAM_BITS[codec]), np.uint8)
    res = np.zeros((S, F, 6), np.int32)
    d = np.zeros(88, np.uint8)
    r = np.zeros(5, np.int32)
    for s in range(S):
        for f in range(F):
            fr = np.ascontiguousarray(frames[s, f])
            res[s, f, 0] = o.mbo_decode_frame(codec, 0, T._ptr(fr), T._ptr(d), T._ptr(r))
            res[s, f, 1:] = r
            bits[s, f] = d[:T.PARAM_BITS[codec]]
    return bits, res


@pytest.fixture(scope="module")
def knob_case(pkg, tmp_path_factory):
    rng = np.random.default_rng(0x6B1B)
    frames = T.mixed_frames(3, KS, 8, 0x6B13)
    bits, res = _oracle_decode(3, frames)
    seeds = T.stream_seeds(KM, 0x6B6)
    slots = rng.permutation(KM)[:KS].astype(np.int32)
    slots[8900], slots[4000], slots[6000] = slots[100], -1, KM
    accepted = np.ones(KS, bool)
    accepted[[8900, 4000, 6000]] = False
    idle = np.setdiff1d(np.arange(KM), slots[accepted]).astype(np.int32)
    inp = str(tmp_path_factory.mktemp("dataknobs") / "in.npz")
    np.savez(inp, max_streams=KM, first_stream=KFIRST, seeds=seeds, bits=bits, results=res, cuts=np.array(KCUTS),
             slots=slots, accepted=accepted, idle_slots=idle)
    sd = seeds[KFIRST:KFIRST + KS]
    want = T.run_cpu(T.load_oracle().mbo_run, 3, 0, frames, sd, n_threads=16)
    want["rng"] = T.oracle_rng_words(3, 0, frames, sd, n_threads=16)
    return dict(inp=inp, want=want, accepted=accepted, res_in=res)


@pytest.mark.parametrize("name,knobs", KSETTINGS, ids=[s[0] for s in KSETTINGS])
def test_data_indexed_under_knobs_equals_the_oracle(knob_case, tmp_path, monkeypatch, name, knobs):
    from test_gpu_knobs import _diff, _expected_launches
    monkeypatch.setattr(T, "KNOB_CHILD", CHILD)
    out = str(tmp_path / "out.npz")
    log = T.run_knob_child(["run", knob_case["inp"], out], knobs, timeout=900)
    z = np.load(out)
    meta = json.loads(str(z["meta"]))
    assert {k: v for k, v in meta["env"].items() if k in T.KNOBS} == {k: str(v) for k, v in knobs.items()}
    assert meta["kernel_path"] == (0 if knobs.get("MBE_B200_SPLIT") == 0 else 1)
    print("\n%s\n%s" % (name, log))
    failures = []
    for c in meta["calls"]:
        lo, hi = _expected_launches(c, meta, knobs)
        if not lo <= c["launches"] <= hi or (meta["kernel_path"] == 1 and (c["launches"] - c["indexed"]) % 3):
            failures.append("%s, %d x %d frames: %d launches, expected %d..%d" % (c["row"], c["n"], c["frames"],
                                                                                c["launches"], lo, hi))
    ok, w = knob_case["accepted"], knob_case["want"]
    res_in = knob_case["res_in"]
    for row in meta["rows"]:
        for k in ("pcm", "pcmf", "results"):
            _diff(failures, row + " " + k, z[row + "." + k][ok], w[k][ok])
        res = z[row + ".results"][~ok]
        _diff(failures, row + " rejected status", res[..., 0], np.full(res.shape[:-1], -1, np.int32))
        _diff(failures, row + " rejected result echo", res[..., 1:], res_in[~ok][..., 1:])
        for k in ("pcm", "pcmf"):
            _diff(failures, row + " rejected " + k, z[row + "." + k][~ok], np.zeros_like(z[row + "." + k][~ok]))
        _diff(failures, row + " state", z[row + ".state"], w["state"][ok])
        _diff(failures, row + " rng", z[row + ".rng"], w["rng"][ok])
        _diff(failures, row + " idle state", z[row + ".idle_state_after"], z[row + ".idle_state_before"])
        _diff(failures, row + " idle rng", z[row + ".idle_rng_after"], z[row + ".idle_rng_before"])
    z.close()
    os.remove(out)
    assert not failures, "%s:\n  %s" % (name, "\n  ".join(failures))
