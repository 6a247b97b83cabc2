"""Does an indexed call cost more than a contiguous one?  IMBE 7200x4400 hard, 50 frames, a context of 1 048 576 slots,
device-resident (mbe_b200_process_frames_dev against mbe_b200_process_indexed_dev over the same number of streams, the
slots a random permutation / a random scattered subset), and the host-pointer call end to end at 1 048 576 streams.
CUDA events for the device calls, a host clock around the (synchronous) host calls; every shape warmed up, A and B
alternated, median and spread of the repetitions.  Writes one JSON file with the card's name and power limit.

    python tools/gpu_indexed_probe.py --out profiles/indexed_probe_b200.json [--reps 7]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from __graft_entry__ import load_package  # noqa: E402

MAX_STREAMS, F, CODEC, FBITS = 1 << 20, 50, 0, 184


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = "unavailable (%s)" % e
    return dict(gpu=name, power_limit_and_max_sm_clock=q)


def stats(xs):
    xs = sorted(xs)
    return dict(median_ms=float(np.median(xs)), min_ms=xs[0], max_ms=xs[-1],
                spread_pct=100.0 * (xs[-1] - xs[0]) / float(np.median(xs)), runs_ms=xs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    pkg = load_package()
    dev = torch.device("cuda", 0)
    dec = pkg.Decoder(max_streams=MAX_STREAMS, device=0)
    dec.init_streams(0, MAX_STREAMS, np.arange(MAX_STREAMS, dtype=np.uint32) + 0xC0FFEE)
    gen = torch.Generator(device=dev)
    gen.manual_seed(0x1D)
    d_frames = torch.randint(0, 2, (MAX_STREAMS, F, FBITS), dtype=torch.uint8, device=dev, generator=gen)
    d_pcm = torch.empty((MAX_STREAMS, F, 160), dtype=torch.int16, device=dev)
    d_res = torch.empty((MAX_STREAMS, F, 6), dtype=torch.int32, device=dev)
    rng = np.random.default_rng(0x1D)
    slot_lists = {MAX_STREAMS: rng.permutation(MAX_STREAMS).astype(np.int32),
                  131072: rng.choice(MAX_STREAMS, 131072, replace=False).astype(np.int32)}
    d_slots = {n: torch.from_numpy(s).to(dev) for n, s in slot_lists.items()}
    st = torch.cuda.Stream(dev)   # (not the legacy default stream: a NULL stream selects the context's own stream)
    torch.cuda.synchronize()

    def contiguous(n):
        dec.process_frames_dev(CODEC, 0, 0, n, F, d_frames.data_ptr(), d_pcm.data_ptr(), d_results=d_res.data_ptr(),
                               cuda_stream=st.cuda_stream)

    def indexed(n):
        dec.process_indexed_dev(CODEC, pkg.INPUT_HARD, d_slots[n].data_ptr(), n, F, d_frames.data_ptr(), d_pcm.data_ptr(),
                                d_results=d_res.data_ptr(), cuda_stream=st.cuda_stream)

    def dev_ms(fn, n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        fn(n)
        b.record(st)
        b.synchronize()
        return a.elapsed_time(b)

    out = dict(card=card(), workload=dict(codec="imbe7200x4400", input="hard", frames=F, context_slots=MAX_STREAMS,
                                          kernel_path=dec.kernel_path(), outputs="int16 PCM + results"),
               device={}, host={})
    for n in (MAX_STREAMS, 131072):
        for fn in (contiguous, indexed):
            fn(n)
            fn(n)
        torch.cuda.synchronize()
        t = dict(contiguous=[], indexed=[])
        for _ in range(args.reps):
            t["contiguous"].append(dev_ms(contiguous, n))
            t["indexed"].append(dev_ms(indexed, n))
        out["device"][str(n)] = {k: stats(v) for k, v in t.items()}
        c, i = out["device"][str(n)]["contiguous"]["median_ms"], out["device"][str(n)]["indexed"]["median_ms"]
        out["device"][str(n)]["indexed_over_contiguous"] = i / c
        out["device"][str(n)]["mframes_per_s"] = dict(contiguous=n * F / c / 1e3, indexed=n * F / i / 1e3)
        print("device n=%d: contiguous %.2f ms, indexed %.2f ms (x%.4f)" % (n, c, i, i / c), flush=True)

    # host-pointer calls end to end, pinned buffers
    n = MAX_STREAMS
    h_frames = torch.empty((n, F, FBITS), dtype=torch.uint8, pin_memory=True)
    h_frames.copy_(d_frames)
    del d_pcm, d_res
    h_pcm = torch.empty((n, F, 160), dtype=torch.int16, pin_memory=True)
    h_res = torch.empty((n, F, 6), dtype=torch.int32, pin_memory=True)
    lib, h = dec.lib, dec.h
    slots = slot_lists[n]
    import ctypes
    vp = ctypes.c_void_p
    pf, pp, pr = (vp(x.data_ptr()) for x in (h_frames, h_pcm, h_res))

    def h_contiguous():
        assert lib.mbe_b200_process_frames(h, CODEC, 0, 0, n, F, pf, pp, None, pr, None) == 0

    def h_indexed():
        assert lib.mbe_b200_process_indexed(h, CODEC, pkg.INPUT_HARD, slots.ctypes.data_as(vp), n, F, pf, pp, None, pr,
                                            None) == 0

    for fn in (h_contiguous, h_indexed):
        fn()
    t = dict(contiguous=[], indexed=[])
    for _ in range(args.reps):
        for k, fn in (("contiguous", h_contiguous), ("indexed", h_indexed)):
            t0 = time.perf_counter()
            fn()
            t[k].append((time.perf_counter() - t0) * 1e3)
    out["host"][str(n)] = {k: stats(v) for k, v in t.items()}
    c, i = out["host"][str(n)]["contiguous"]["median_ms"], out["host"][str(n)]["indexed"]["median_ms"]
    out["host"][str(n)]["indexed_over_contiguous"] = i / c
    print("host n=%d: contiguous %.1f ms, indexed %.1f ms (x%.4f)" % (n, c, i, i / c), flush=True)
    out["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    dec.close()


if __name__ == "__main__":
    main()
