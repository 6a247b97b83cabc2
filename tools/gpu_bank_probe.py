"""How full are the bank kernel's 32-slot passes, and what does the kernel cost per frame?  Runs the single-GPU bench
workloads of BASELINE.json configs[2] (IMBE 7200x4400 hard, 1 048 576 streams), configs[1] (AMBE+2 hard, 65 536 streams)
and configs[3] (AMBE 3600x2400 tone / unvoiced-only / voice frames, 262 144 streams), 50 frames per launch,
device-resident on the default (multi-kernel) path, with bench.py's input frames and stream seeds.  For the current build
it reports, from mbe_b200_kernel_timing (CUDA-event pairs around every launch, and the counters the bank kernel keeps
itself):

  * the bank kernel's bracketed event time per frame of the workload, next to the step time per frame;
  * oscillator slots, phase-interpolated harmonics and 32-slot passes per synthesised frame;
  * lane fill = slots / (32 x passes);
  * the card's name, power limit and SM clock, read in the same run.

    python tools/gpu_bank_probe.py --out profiles/bank_probe_b200.json [--steps 3] [--warmup 1]

MBE_B200_LIB selects another build of the library (an A/B against the in-tree one)."""
import argparse
import ctypes
import importlib.util
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from __graft_entry__ import load_package  # noqa: E402
import bench  # noqa: E402  (input generation only: the workload is bench.py's own)

_spec = importlib.util.spec_from_file_location("mbe_b200_sharding", os.path.join(ROOT, "mbelib-neo_b200", "sharding.py"))
sharding = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(sharding)

F = 50


def card():
    q = "unavailable"
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = "unavailable (%s)" % e
    return dict(gpu=torch.cuda.get_device_name(0), power_limit_sm_clock_max_sm_clock=q)


def kernel_timing(dec):
    """mbe_b200_kernel_timing with all four counters ([3]: the bank kernel's passes), straight through the C-ABI."""
    ms = (ctypes.c_double * 3)()
    n = (ctypes.c_longlong * 3)()
    cnt = (ctypes.c_ulonglong * 4)()
    assert dec.lib.mbe_b200_kernel_timing(dec.h, ms, n, cnt) == 0
    return list(ms), list(n), list(cnt)


def probe(pkg, config, steps, warmup):
    (codec_name, kind), = bench.CONFIGS[config]["parts"]
    codec, S = bench.CODEC_IDS[codec_name], bench.CONFIGS[config]["streams"]
    name = "configs[%d]" % config
    dev = torch.device("cuda", 0)
    dec = pkg.Decoder(max_streams=S, device=0)
    dec.init_streams(0, S, sharding.stream_seeds(0, S))
    if kind == "hard":
        frames = bench.counter_bits_torch(codec, 0, S, F, dev)
    else:   # as bench.py builds it: 128 distinct seeded streams tiled over the range
        base = torch.from_numpy(bench.part_frames_numpy(codec, kind, 0, 128, F)).to(dev)
        frames = base[torch.arange(S, device=dev) % 128].contiguous()
    pcm = torch.empty((S, F, 160), dtype=torch.int16, device=dev)
    res = torch.empty((S, F, 6), dtype=torch.int32, device=dev)
    st = torch.cuda.Stream(dev)

    def step():
        dec.process_frames_dev(codec, 0, 0, S, F, frames.data_ptr(), pcm.data_ptr(), 0, res.data_ptr(), 0, st.cuda_stream)

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dec.set_kernel_timing(True)
    a.record(st)
    for _ in range(steps):
        step()
    b.record(st)
    b.synchronize()
    ms, launches, cnt = kernel_timing(dec)
    dec.set_kernel_timing(False)
    step_ms = a.elapsed_time(b) / steps
    slots, interp, synth, passes = cnt
    n = S * F * steps
    out = dict(codec=codec_name, input=kind, streams=S, frames=F, steps=steps,
               kernel_path=dec.kernel_path(), step_ms=step_ms, mframes_per_s=S * F / step_ms / 1e3,
               ns_per_frame=dict(step=step_ms * 1e6 / (S * F), bank=ms[1] * 1e6 / n, parameter=ms[0] * 1e6 / n,
                                 unvoiced=ms[2] * 1e6 / n),
               bank_launches=launches[1], synthesised_frames=synth,
               per_synthesised_frame=dict(slots=slots / max(1, synth), interpolated=interp / max(1, synth),
                                          passes=passes / max(1, synth)),
               lane_fill=slots / max(1, 32 * passes))
    print("%s: %.1f M frames/s, bank %.3f ns/frame, slots %.2f, passes %.3f per frame, fill %.4f" % (
        name, out["mframes_per_s"], out["ns_per_frame"]["bank"], out["per_synthesised_frame"]["slots"],
        out["per_synthesised_frame"]["passes"], out["lane_fill"]), flush=True)
    dec.close()
    del frames, pcm, res
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()
    pkg = load_package()
    out = dict(library=os.environ.get("MBE_B200_LIB") or "in-tree", card=card(), workloads={})
    for config in (2, 1, 3):
        out["workloads"]["configs[%d]" % config] = probe(pkg, config, args.steps, args.warmup)
    out["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
