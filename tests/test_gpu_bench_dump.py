"""bench.py --dump-outputs on the GPU: the dumped sample is what the timed path returned in its last step (checked against the
CPU oracle fed the same frames for warmup + steps passes), a rerun with the same arguments dumps the same arrays, --steps
sets the number of timed steps, and on a multi-part workload larger than the sample every part's sampled stream ids name
the streams whose outputs were written."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import mbe_testlib as T
from __graft_entry__ import ROOT

pytestmark = pytest.mark.gpu

CODEC, S, F, WARMUP = T.AMBE2450, 64, 50, 1


def _run_bench(out_dir, args):
    args = args + ["--no-cpu-baseline", "--no-e2e", "--dump-outputs", out_dir]
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])


def _load(out_dir, part):
    return {k: np.load(os.path.join(out_dir, "%s_%s.npy" % (part, k))) for k in ("streams", "pcm", "results")}


def _bench(out_dir, steps):
    line = _run_bench(out_dir, ["--codec", T.CODEC_NAMES[CODEC], "--streams", str(S), "--frames", str(F), "--warmup", str(WARMUP),
                                "--steps", str(steps)])
    return line, _load(out_dir, "%s_hard" % T.CODEC_NAMES[CODEC])


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    return b


def _expected_results(results):
    res = results.astype(np.int64)
    res[..., 5] &= 0xffffffff
    return res.astype(np.float64)


def test_dump_is_the_last_timed_step(tmp_path):
    b = _bench_module()
    frames = b.counter_bits_numpy(CODEC, 0, S, F)
    launches = {}
    for steps in (2, 3):
        line, d = _bench(str(tmp_path / ("s%d" % steps)), steps)
        assert line["steps"] == steps
        launches[steps] = line["gpu_launches"]
        assert d["streams"].dtype == np.float64 and d["pcm"].dtype == np.float32 and d["results"].dtype == np.float64
        assert np.array_equal(d["streams"], np.arange(S))          # fewer streams than the sample size: all of them
        assert d["pcm"].shape == (S, F, 160) and d["results"].shape == (S, F, 6)
        # every step decodes the same frames, so the last step is frames F * (warmup + steps - 1) ... of one long stream
        want = T.run_cpu(T.load_oracle().mbo_run, CODEC, 0, np.concatenate([frames] * (WARMUP + steps), axis=1),
                         T.stream_seeds(S), want_float=False, want_state=False)
        assert np.array_equal(d["results"], _expected_results(want["results"][:, -F:]))
        diff = np.abs(d["pcm"] - want["pcm"][:, -F:].astype(np.float32))
        assert diff.max() <= 2 and (diff == 0).mean() >= 0.9999, (diff.max(), (diff == 0).mean())
        if steps == 2:
            first = d
    assert launches[2] > 0 and launches[3] * 2 == launches[2] * 3
    _, again = _bench(str(tmp_path / "again"), 2)
    for k in first:
        assert np.array_equal(first[k], again[k]), k


def test_sampled_streams_of_every_part(tmp_path):
    """BASELINE configs[4] (three codecs, soft-decision input) at 3 x 1000 streams: each part dumps a seeded sample of
    DUMP_MAX_STREAMS of its streams, and the ids it records are the global streams whose outputs were written."""
    b = _bench_module()
    n_frames, total = 8, 3000
    out = str(tmp_path / "c4")
    line = _run_bench(out, ["--config", "4", "--streams", str(total), "--frames", str(n_frames), "--warmup", "0", "--steps", "1"])
    assert line["steps"] == 1
    size = sum(os.path.getsize(os.path.join(out, f)) for f in os.listdir(out))
    assert len(os.listdir(out)) == 9 and size <= b.DUMP_BUDGET_BYTES
    for p, (name, kind) in enumerate(b.CONFIGS[4]["parts"]):
        codec = b.CODEC_IDS[name]
        d = _load(out, "%s_%s" % (name, kind))
        ids = d["streams"].astype(np.int64)
        lo, hi = total * p // 3, total * (p + 1) // 3
        assert len(ids) == b.DUMP_MAX_STREAMS < hi - lo and np.all(np.diff(ids) > 0) and lo <= ids[0] and ids[-1] < hi
        assert np.array_equal(d["streams"], ids.astype(np.float64))
        # softch input: 128 seeded streams tiled over the global stream ids; one step from freshly seeded state
        frames = b.part_frames_numpy(codec, kind, 0, 128, n_frames)[ids % 128]
        seeds = ((ids + 0xC0FFEE) & 0xffffffff).astype(np.uint32)
        want = T.run_cpu(T.load_oracle().mbo_run, codec, 1, frames, seeds, n_threads=os.cpu_count() or 1,
                         want_float=False, want_state=False)
        assert np.array_equal(d["results"], _expected_results(want["results"])), name
        diff = np.abs(d["pcm"] - want["pcm"].astype(np.float32))
        assert diff.max() <= 2 and (diff == 0).mean() >= 0.9999, (name, diff.max(), (diff == 0).mean())
