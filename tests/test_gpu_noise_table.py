"""The unvoiced kernel's noise spectrum table (mbe_split.cuh, DESIGN 4.5): a synthesis frame whose overlap is the natural one of
its generator state takes its forward noise spectrum from the context's table, any other frame computes it.  Both give the
same bits, so MBE_B200_NOISE_TABLE=0 must change nothing but the counters.  The knob is read once per process, so every run
happens in a child process (tests/helpers/noise_table_child.py).

Imported states exercise the check: overlaps and seeds that are not each other's natural pair must fall back and still equal
the CPU oracle; a natural overlap under a seed that truncates to the same generator state must hit."""
import ctypes
import importlib.util
import os
import subprocess
import sys

import numpy as np
import pytest

import mbe_testlib as T
from __graft_entry__ import load_package

pytestmark = pytest.mark.gpu

CHILD = os.path.join(T.ROOT, "tests", "helpers", "noise_table_child.py")
SEED_W, OV_W = 554, 555           # noiseSeed and noiseOverlap[96] words of an mbe_parms image (mbe_common.cuh)
S, F0, F1 = 96, 5, 6              # imported-state cases: streams, frames before the export, frames after the import


def _child(cases, table, tmp_path):
    inp, outp = str(tmp_path / ("in%d.npz" % table)), str(tmp_path / ("out%d.npz" % table))
    np.savez(inp, **{n + "." + k: v for n, c in cases.items() for k, v in c.items()})
    env = {k: v for k, v in os.environ.items() if k not in T.KNOBS and k != "MBE_B200_NOISE_TABLE"}
    env["MBE_B200_NOISE_TABLE"] = str(table)
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [CHILD, inp, outp]
    p = subprocess.run(cmd, env=env, timeout=900, capture_output=True, text=True)
    assert p.returncode == 0, p.stdout[-4000:] + p.stderr[-4000:]
    z = np.load(outp)
    return {n: {k: z[n + "." + k] for k in ("pcm", "pcmf", "results", "state", "counters")} for n in cases}


def _same(a, b, what):
    for k in ("pcm", "pcmf", "results", "state"):
        assert np.array_equal(a[k].view(np.uint8), b[k].view(np.uint8)), "%s: %s differs" % (what, k)


def _tones_frames(n, f, seed):
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(T.ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench.tone_unvoiced_frames(n, f, seed)


def test_table_on_equals_table_off(tmp_path):
    """Every codec on random frames, and configs[3]-shaped AMBE 3600x2400 frames (a third of them unvoiced-only), with the
    table and without it: PCM (int16 and float), results and end states equal bit for bit."""
    cases = {}
    for codec in range(4):
        cases["c%d" % codec] = dict(codec=np.int32(codec), frames=T.random_hard_frames(codec, 384, 12, 0x7AB + codec),
                                    seeds=T.stream_seeds(384, 0x5EED + codec))
    cases["tones"] = dict(codec=np.int32(2), frames=_tones_frames(384, 12, 0x70E5), seeds=T.stream_seeds(384, 0x70))
    on, off = _child(cases, 1, tmp_path), _child(cases, 0, tmp_path)
    for n in cases:
        _same(on[n], off[n], n)
        hit, miss = on[n]["counters"]
        hit0, miss0 = off[n]["counters"]
        print("%s: %d of %d synthesised frames from the table" % (n, hit, hit + miss))
        assert hit0 == 0 and miss0 > 0
        assert hit + miss == miss0
        assert hit > miss   # after its first synthesised frame a stream's overlap is natural


def _oracle_continue(codec, frames, state, rng):
    """The oracle from imported states: mbo_process_frame frame by frame (mbo_run's per-frame body)."""
    o = T.load_oracle()
    vp = ctypes.c_void_p
    o.mbo_process_frame.argtypes = [ctypes.c_int, ctypes.c_int] + [vp] * 8
    o.mbo_process_frame.restype = ctypes.c_int
    o.mbo_float_to_short.argtypes = [vp, vp]
    n, f = frames.shape[0], frames.shape[1]
    out = dict(pcm=np.zeros((n, f, 160), np.int16), pcmf=np.zeros((n, f, 160), np.float32),
               state=np.ascontiguousarray(state.copy()))
    rng = np.ascontiguousarray(rng.copy())
    for s in range(n):
        st = out["state"][s]
        for k in range(f):
            pf, ps = np.zeros(160, np.float32), np.zeros(160, np.int16)
            res, bits = np.zeros(16, np.int32), np.zeros(128, np.uint8)
            fr = np.ascontiguousarray(frames[s, k])
            ret = o.mbo_process_frame(codec, 0, T._ptr(pf), T._ptr(res), T._ptr(fr), T._ptr(bits), T._ptr(st[0]),
                                      T._ptr(st[1]), T._ptr(st[2]), T._ptr(rng[s]))
            if ret >= 0:
                o.mbo_float_to_short(T._ptr(pf), T._ptr(ps))
                out["pcm"][s, k], out["pcmf"][s, k] = ps, pf
    return out


def test_imported_states_fall_back_or_hit(tmp_path):
    """IMBE 7200x4400: states after F0 frames (oracle), edited in cur_mp of every stream that has left its cold start, then
    imported and decoded for F1 more frames.  Must fall back: random overlaps, a natural overlap with one word one ulp off,
    seeds that truncate to another generator state (non-integer, >= 53125), -0.0, negative seeds.  Must hit: the natural
    overlap under seed + 0.25 and under seed + 53125 (the same generator state).  Every case equals the oracle.  A case adds
    fallbacks over the unedited import, at most one per edited stream; after a negative seed (a cold start, which leaves a
    zero overlap that is not the natural one of its new seed) only the increase is asserted."""
    codec = 0
    frames = T.random_hard_frames(codec, S, F0 + F1, 0x1A7E)
    seeds = T.stream_seeds(S, 0x1A)
    warm = T.run_cpu(T.load_oracle().mbo_run, codec, 0, frames[:, :F0], seeds)
    rng = T.oracle_rng_words(codec, 0, frames[:, :F0], seeds)
    base = warm["state"]
    f32 = lambda st: st.view(np.float32).reshape(S, 3, -1)
    seed0 = f32(base)[:, 0, SEED_W].copy()
    live = seed0 >= 0.0
    assert live.sum() >= S // 2
    r = np.random.default_rng(0xED17)

    def edit(fn):
        st = base.copy()
        v = f32(st)
        for s in np.nonzero(live)[0]:
            fn(v[s, 0], s)
        return st

    def set_seed(x):
        def fn(p, s):
            p[SEED_W] = np.float32(x(seed0[s]))
        return fn

    def rand_ov(p, s):
        p[OV_W:OV_W + 96] = r.integers(0, 53125, 96).astype(np.float32)

    def ulp(p, s):
        w = p[OV_W:OV_W + 96].view(np.uint32)
        w[int(r.integers(0, 96))] += 1

    fallback = dict(random_overlap=edit(rand_ov), ulp_overlap=edit(ulp),
                    seed_fraction=edit(set_seed(lambda x: x + 1.5)), seed_large=edit(set_seed(lambda x: x + 106257.0)),
                    seed_minus_zero=edit(set_seed(lambda x: -0.0)), seed_negative=edit(set_seed(lambda x: -5.0)))
    hit = dict(seed_quarter=edit(set_seed(lambda x: x + 0.25)), seed_period=edit(set_seed(lambda x: x + 53125.0)))
    states = dict(natural=base, **fallback, **hit)
    # -0.0 is generator state 0: a stream whose natural state is 0 would hit
    assert not np.any(seed0[live] == 0.0)
    cases = {n: dict(codec=np.int32(codec), frames=frames[:, F0:], seeds=seeds, state=st, rng=rng) for n, st in states.items()}
    on, off = _child(cases, 1, tmp_path), _child(cases, 0, tmp_path)
    n_edit = int(live.sum())
    base_miss = on["natural"]["counters"][1]
    for n, st in states.items():
        want = _oracle_continue(codec, frames[:, F0:], st, rng)
        for k in ("pcm", "pcmf", "state"):
            assert np.array_equal(on[n][k].view(np.uint8), want[k].view(np.uint8)), "%s: %s differs from the oracle" % (n, k)
        _same(on[n], off[n], n)
        h, m = on[n]["counters"]
        assert h + m == off[n]["counters"][1] and off[n]["counters"][0] == 0
        print("%s: %d hits, %d fallbacks (unedited import: %d fallbacks)" % (n, h, m, base_miss))
        if n in fallback:
            assert 0 < m - base_miss and (n == "seed_negative" or m - base_miss <= n_edit), n
        elif n in hit:
            assert m == base_miss, n


def test_table_built_on_one_caller_stream_orders_a_call_on_another():
    """The table is built on the stream of a context's first multi-kernel launch.  A second call on another caller stream,
    cut into more stream ranges than the first (so that it forks onto internal streams the first call never used), must not
    read the table before that build has run, even when the first stream still has earlier work queued ahead of it.  Its
    outputs equal the same decode repeated once everything has finished."""
    import torch
    pkg = load_package()
    dev = torch.device("cuda", 0)
    # one full range (10 656 streams x 50 frames by default) for the first call and three smaller ones for the second, so that
    # the second call reuses the first one's descriptor buffer as it is (growing it would synchronise the device)
    codec, S1, S2, F = 0, 10000, 3 * 9990, 50
    f1 = torch.from_numpy(T.random_hard_frames(codec, S1, F, 0x0DE1)).to(dev)
    f2 = torch.from_numpy(T.random_hard_frames(codec, S2, F, 0x0DE2)).to(dev)
    pcm1 = torch.empty((S1, F, 160), dtype=torch.int16, device=dev)
    pcm2 = torch.empty((S2, F, 160), dtype=torch.int16, device=dev)
    ref2 = torch.empty_like(pcm2)
    seeds2 = T.stream_seeds(S2, 0x0DE)
    dec = pkg.Decoder(max_streams=S1 + S2, device=0)
    dec.set_kernel_path(1)
    dec.init_streams(0, S1, T.stream_seeds(S1, 0x0D))
    dec.init_streams(S1, S2, seeds2)
    x, y = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    torch.cuda.synchronize()
    with torch.cuda.stream(x):
        torch.cuda._sleep(1 << 30)      # earlier work of the caller on stream x, ahead of the table build
    dec.process_frames_dev(codec, 0, 0, S1, F, f1.data_ptr(), pcm1.data_ptr(), cuda_stream=x.cuda_stream)
    n0 = dec.launches
    dec.process_frames_dev(codec, 0, S1, S2, F, f2.data_ptr(), pcm2.data_ptr(), cuda_stream=y.cuda_stream)
    assert dec.launches - n0 == 9, "the second call should run in three stream ranges"
    torch.cuda.synchronize()
    dec.init_streams(S1, S2, seeds2)
    dec.process_frames_dev(codec, 0, S1, S2, F, f2.data_ptr(), ref2.data_ptr(), cuda_stream=y.cuda_stream)
    torch.cuda.synchronize()
    assert torch.equal(pcm2, ref2)
    dec.close()
