"""bench.py contract checks that need no GPU: the reference arm (`--impl reference`) runs the unmodified reference's CPU
build from oracle/_ref (or the oracle port when it is absent) and prints one JSON line with the keys the driver reads;
the default arm refuses to run without a CUDA device instead of falling back to the CPU."""
import json
import os
import subprocess
import sys

import pytest

from __graft_entry__ import ROOT


def _run(args, timeout=600):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=timeout)


def test_reference_arm_prints_the_contract_line():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "1"])
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["metric"] == "decoded frames/sec" and line["unit"] == "frames/s"
    assert line["higher_is_better"] is True and line["scaling"] == "strong" and line["gpu_launches"] == 0
    assert line["value"] > 0 and line["ms_per_step"] > 0
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # default workload = BASELINE.json configs[2]: IMBE 7200x4400, 1M streams sharded over the GPUs
    assert "IMBE 7200x4400" in line["config"]["workload"] and line["config"]["baseline_config"] == "configs[2]"
    assert line["config"]["total_streams"] == 1048576 and line["config"]["frames_per_stream"] == 50


def test_other_configs_and_custom_workloads_parse():
    for args, part in ((["--config", "1"], "ambe3600x2450/hard"), (["--codec", "ambe3600x2400", "--streams", "64"], "ambe3600x2400/hard")):
        r = _run(["--impl", "reference", "--steps", "1", "--warmup", "1"] + args)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
        assert line["config"]["parts"] == [part] and line["scaling"] == "weak" and line["value"] > 0


def test_zero_steps_are_refused():
    r = _run(["--impl", "reference", "--steps", "0", "--warmup", "1"])
    assert r.returncode != 0 and "--steps" in r.stderr


def test_counter_based_input_is_the_same_on_both_arms():
    """the numpy generator (CPU arm) and the torch generator (GPU arm, run here on the CPU) give identical bits"""
    import importlib.util
    import numpy as np
    import torch
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    for codec in (0, 1, 3):
        a = b.counter_bits_numpy(codec, 1000003, 37, 5)
        t = b.counter_bits_torch(codec, 1000003, 37, 5, torch.device("cpu"), chunk=16).numpy()
        assert a.shape == (37, 5, b.FRAME_BITS[codec]) and np.array_equal(a, t)
        assert 0.45 < a.mean() < 0.55
        # a shard sees the same bits as the whole: stream 1000010 from two different windows
        assert np.array_equal(b.counter_bits_numpy(codec, 1000010, 1, 5)[0], a[7])


def test_reference_arm_on_other_ranks_exits_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_default_arm_has_no_cpu_path():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    r = _run(["--steps", "1", "--warmup", "1"], timeout=300)
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)
