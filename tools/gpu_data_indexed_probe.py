"""Does an indexed parameter-bit call cost more than a contiguous one, and what does the pipelined, packed host call gain?
IMBE 7200x4400 parameter bits with their decode contexts (the decode of valid random frames: a pool of 2 048 frames
encoded from random parameters, decoded on the device, drawn at random for every stream-frame), 50 frames, a context of
1 048 576 slots, the multi-kernel path, int16 PCM plus results.
  device: mbe_b200_process_data_dev against mbe_b200_process_data_indexed_dev over the same number of streams (the slots
          a random permutation of all 1 048 576 / 131 072 scattered slots), CUDA events on one caller stream;
  host:   mbe_b200_process_data (contiguous, one copy-in / kernel / copy-out), mbe_b200_process_data_indexed one byte per
          bit and packed (pipelined), pinned buffers, a host clock around the synchronous calls.
Every shape is warmed up, the variants alternate, median and spread of the repetitions.  Writes one JSON file with the
card's name, power limit and maximum SM clock.

    python tools/gpu_data_indexed_probe.py --out profiles/data_indexed_probe_b200.json [--reps 7]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from __graft_entry__ import load_package  # noqa: E402
import mbe_testlib as T  # noqa: E402

MAX_STREAMS, F, CODEC, PBITS, POOL = 1 << 20, 50, 0, 88, 2048


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
    dec.set_kernel_path(1)
    dec.init_streams(0, MAX_STREAMS, np.arange(MAX_STREAMS, dtype=np.uint32) + 0xC0FFEE)

    # valid frames from random parameters, decoded by the library: parameter bits + decode contexts
    rng = np.random.default_rng(0xDA7A)
    params = rng.integers(0, 2, size=(POOL, PBITS), dtype=np.uint8)
    params[:, CODEC] = 0
    frames = np.stack([T.encode_imbe7200_frame(p).reshape(-1) for p in params])
    pool_bits, pool_res = dec.decode_frames(CODEC, frames)
    gen = torch.Generator(device=dev)
    gen.manual_seed(0xDA7A)
    pick = torch.randint(0, POOL, (MAX_STREAMS, F), device=dev, generator=gen)
    d_bits = torch.from_numpy(pool_bits).to(dev)[pick]                                            # [S][F][88]
    d_packed = torch.from_numpy(pkg.pack_params(CODEC, pool_bits)).to(dev)[pick]                 # [S][F][11]
    d_ctx = torch.from_numpy(np.ascontiguousarray(pool_res).view(np.int32).reshape(POOL, 6)).to(dev)[pick]
    del pick
    d_res = d_ctx.clone()
    d_pcm = torch.empty((MAX_STREAMS, F, 160), dtype=torch.int16, device=dev)
    slot_lists = {MAX_STREAMS: rng.permutation(MAX_STREAMS).astype(np.int32),
                  131072: rng.choice(MAX_STREAMS, 131072, replace=False).astype(np.int32)}
    d_slots = {n: torch.from_numpy(s).to(dev) for n, s in slot_lists.items()}
    st = torch.cuda.Stream(dev)   # (not the legacy default stream: a NULL stream selects the context's own stream)
    torch.cuda.synchronize()
    lib, h, vp = dec.lib, dec.h, ctypes.c_void_p

    def contiguous(n):
        assert lib.mbe_b200_process_data_dev(h, CODEC, 0, n, F, vp(d_bits.data_ptr()), vp(d_res.data_ptr()),
                                             vp(d_pcm.data_ptr()), None, vp(st.cuda_stream)) == 0

    def indexed(n):
        dec.process_data_indexed_dev(CODEC, False, d_slots[n].data_ptr(), n, F, d_bits.data_ptr(), d_res.data_ptr(),
                                     d_pcm.data_ptr(), cuda_stream=st.cuda_stream)

    def dev_ms(fn, n):
        with torch.cuda.stream(st):
            d_res.copy_(d_ctx)      # every call decodes with the same contexts (the results are IN/OUT)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        fn(n)
        b.record(st)
        b.synchronize()
        return a.elapsed_time(b)

    out = dict(card=card(), workload=dict(codec="imbe7200x4400", input="parameter bits + decode context (decode of valid "
                                          "random frames)", frames=F, context_slots=MAX_STREAMS,
                                          kernel_path=dec.kernel_path(), outputs="int16 PCM + results"),
               device={}, host={})
    for n in (MAX_STREAMS, 131072):
        for fn in (contiguous, indexed):
            dev_ms(fn, n)
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
    h_bits = torch.empty((n, F, PBITS), dtype=torch.uint8, pin_memory=True)
    h_bits.copy_(d_bits)
    h_packed = torch.empty((n, F, 11), dtype=torch.uint8, pin_memory=True)
    h_packed.copy_(d_packed)
    h_ctx = d_ctx.cpu()
    del d_bits, d_packed, d_ctx, d_res, d_pcm, d_slots
    torch.cuda.empty_cache()
    h_pcm = torch.empty((n, F, 160), dtype=torch.int16, pin_memory=True)
    h_res = torch.empty((n, F, 6), dtype=torch.int32, pin_memory=True)
    slots = slot_lists[n]
    pb, pk, pp, pr = (vp(x.data_ptr()) for x in (h_bits, h_packed, h_pcm, h_res))
    ps = slots.ctypes.data_as(vp)
    calls = dict(
        contiguous=lambda: lib.mbe_b200_process_data(h, CODEC, 0, n, F, pb, pr, pp, None),
        indexed=lambda: lib.mbe_b200_process_data_indexed(h, CODEC, 0, ps, n, F, pb, pr, pp, None),
        indexed_packed=lambda: lib.mbe_b200_process_data_indexed(h, CODEC, 1, ps, n, F, pk, pr, pp, None))
    for fn in calls.values():
        h_res.copy_(h_ctx)
        assert fn() == 0
    t = {k: [] for k in calls}
    for _ in range(args.reps):
        for k, fn in calls.items():
            h_res.copy_(h_ctx)
            t0 = time.perf_counter()
            assert fn() == 0
            t[k].append((time.perf_counter() - t0) * 1e3)
    out["host"][str(n)] = {k: stats(v) for k, v in t.items()}
    c = out["host"][str(n)]["contiguous"]["median_ms"]
    for k in ("indexed", "indexed_packed"):
        out["host"][str(n)][k + "_over_contiguous"] = out["host"][str(n)][k]["median_ms"] / c
    out["host"][str(n)]["mframes_per_s"] = {k: n * F / out["host"][str(n)][k]["median_ms"] / 1e3 for k in calls}
    print("host n=%d: %s" % (n, {k: round(out["host"][str(n)][k]["median_ms"], 1) for k in calls}), flush=True)
    out["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    dec.close()


if __name__ == "__main__":
    main()
