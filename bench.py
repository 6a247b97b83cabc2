#!/usr/bin/env python
"""bench.py - decoded 20 ms frames/s of the batched IMBE/AMBE decode+synthesis path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 1|2|3|4] [--dump-outputs DIR]

One "step" = one pass of the hot path (frame bits -> ECC -> parameter decode -> synthesis -> int16 PCM) over one batch.
Default workload = BASELINE.json configs[2], the configuration the metric is quoted on: IMBE 7200x4400 hard-decision ECC +
synthesis, 1,048,576 streams x 50 synthetic random-bit frames, the streams SHARDED over the N GPUs (1M / N per rank, "scaling":
"strong"; /root/reference/src/imbe/imbe7200x4400.c:986-1001 is the per-frame call it replaces).  --config 1 / 3 / 4 select the
other BASELINE configs (AMBE+2 65,536 streams per GPU; AMBE 3600x2400 tone / unvoiced-heavy frames, 262,144 streams; the
mixed-codec soft-decision workload, 1M streams, a third per codec); --codec / --streams / --soft ... build a custom single-codec
workload with --streams per GPU (used by the A/B tools).  Streams are independent, so N GPUs run N disjoint stream shards with no
collective on the data path; torch.distributed is used only for the barrier and the max-over-ranks of the timings.

Numbers in the JSON line:
  value        frames/s, whole job, inputs resident in HBM, timed with CUDA events on the launching stream.
  e2e          frames/s through the host-pointer C-ABI call (mbe_b200_process_frames[_packed]): pinned HOST frame bits in,
               int16 PCM + results in HOST memory out, copies inside the timed region; link_ceiling = the same bytes moved
               by plain cudaMemcpyAsync on all ranks at once (what the box's host links allow), frac_of_link = e2e / that.
  roofline     the bound that applies (FP32 issue; parity forbids FMA contraction): algorithmic FLOP per launch / launch time
               against 148 SM x 128 lanes x sampled SM clock; traffic = ncu DRAM bytes per launch; issue_slots = ncu warp
               instructions per frame x frames/s against 148 x 4 schedulers x SM clock (profiles/ncu_constants.json).
  roofline_hbm the HBM view of the same launch (algorithmic bytes / launch time against the measured copy peak).
  cpu_baseline the reference's own CPU build (oracle/_ref, dev-release flags) on the box's host cores, bounded sample of the
               same workload, the SAME counter-based input bits.
`--impl reference` times only that CPU arm.  The CUDA library is mandatory for the default arm: there is no CPU fallback in
the product, and nothing under oracle/ is on the measured GPU path.

--dump-outputs DIR writes what the device-resident arm's last timed step returned, for a fixed seeded sample of rank 0's
streams (at most DUMP_MAX_STREAMS per part, DUMP_BUDGET_BYTES in all), as DIR/<codec>_<input kind>_{streams,pcm,results}.npy:
global stream ids (float64), int16 PCM as float32 [streams][frames][160] and the six mbe_b200_result words as float64
[streams][frames][6].  Inputs and stream seeds depend only on the arguments, so two builds run with the same arguments can be
compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

CODEC_NAMES = {0: "imbe7200x4400", 1: "imbe7100x4400", 2: "ambe3600x2400", 3: "ambe3600x2450"}
CODEC_IDS = {v: k for k, v in CODEC_NAMES.items()}
FRAME_BITS = {0: 184, 1: 168, 2: 96, 3: 96}
# algorithmic FLOP per frame on iid random-bit frames (SURVEY.md 8(d); non-fused, mul = add = 1)
FLOP_PER_FRAME = {0: 84e3, 1: 84e3, 2: 66e3, 3: 61e3}
STATE_BYTES = 7828  # 3 x mbe_parms + 16 B RNG words per stream
RESULT_BYTES = 24
HBM_FALLBACK_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback
INPUT_SEED = 0x4400
DUMP_SEED = 0xD0D0
DUMP_MAX_STREAMS = 512
DUMP_BUDGET_BYTES = 64 << 20

# BASELINE.json configs; a part = (codec, input kind).  Input kinds: "hard" iid random bits (counter-based, identical on the
# CPU and the GPU arm), "tones" configs[3]-shaped frames, "softch" configs[4]-shaped soft-decision frames.
CONFIGS = {
    1: {"parts": [("ambe3600x2450", "hard")], "streams": 65536, "scaling": "weak",
        "what": "configs[1] AMBE+2 3600x2450 hard-decision, 65,536 streams per GPU"},
    2: {"parts": [("imbe7200x4400", "hard")], "streams": 1048576, "scaling": "strong",
        "what": "configs[2] IMBE 7200x4400 hard-decision ECC + synthesis, 1,048,576 streams sharded over the GPUs"},
    3: {"parts": [("ambe3600x2400", "tones")], "streams": 262144, "scaling": "strong",
        "what": "configs[3] AMBE 3600x2400 tone / unvoiced-only / voice frames, 262,144 streams sharded over the GPUs"},
    4: {"parts": [("imbe7200x4400", "softch"), ("imbe7100x4400", "softch"), ("ambe3600x2450", "softch")], "streams": 1048576,
        "scaling": "strong",
        "what": "configs[4] mixed-codec soft-decision (a third of the streams per codec), valid frames with 10% flipped bits, "
                "1,048,576 streams sharded over the GPUs"},
}


def ncu_constants():
    """Per (codec, input kind) constants measured with ncu on this kernel build: executed warp-instructions, FP32 thread
    instructions and DRAM bytes per frame.  Written by tools/ncu_constants.py from the captures of tools/gpu_prof.sh."""
    p = os.path.join(ROOT, "profiles", "ncu_constants.json")
    try:
        with open(p) as f:
            return json.load(f)
    except Exception:
        return {}


def _splitmix64_np(x):
    x = (x + np.uint64(0x9E3779B97F4A7C15))
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return x ^ (x >> np.uint64(31))


def counter_bits_numpy(codec, first_stream, n_streams, n_frames, seed=INPUT_SEED):
    """iid Bernoulli(1/2) channel bits as a pure function of (seed, codec, GLOBAL stream id, frame, bit): bit j of word k of
    splitmix64(seed ^ codec << 56 ^ stream << 24 ^ frame << 8 ^ k) is frame bit 64 k + j.  uint8 [streams][frames][bits]."""
    fb = FRAME_BITS[codec]
    nw = (fb + 63) // 64
    with np.errstate(over="ignore"):
        s = (np.arange(n_streams, dtype=np.uint64) + np.uint64(first_stream))[:, None, None]
        f = np.arange(n_frames, dtype=np.uint64)[None, :, None]
        k = np.arange(nw, dtype=np.uint64)[None, None, :]
        key = np.uint64(seed) ^ (np.uint64(codec) << np.uint64(56)) ^ (s << np.uint64(24)) ^ (f << np.uint64(8)) ^ k
        w = _splitmix64_np(key)
    bits = ((w[..., None] >> np.arange(64, dtype=np.uint64)) & np.uint64(1)).astype(np.uint8)
    return np.ascontiguousarray(bits.reshape(n_streams, n_frames, nw * 64)[:, :, :fb])


def counter_bits_torch(codec, first_stream, n_streams, n_frames, device, seed=INPUT_SEED, chunk=32768):
    """The same bits generated on the device (int64 arithmetic wraps like uint64; right shifts are made logical)."""
    import torch
    fb = FRAME_BITS[codec]
    nw = (fb + 63) // 64
    out = torch.empty((n_streams, n_frames, fb), dtype=torch.uint8, device=device)

    def i64(v):
        v &= (1 << 64) - 1
        return v - (1 << 64) if v >= (1 << 63) else v

    def lsr(x, n):
        return (x >> n) & ((1 << (64 - n)) - 1)

    f = torch.arange(n_frames, dtype=torch.int64, device=device)[None, :, None]
    k = torch.arange(nw, dtype=torch.int64, device=device)[None, None, :]
    sh = torch.arange(64, dtype=torch.int64, device=device)
    for s0 in range(0, n_streams, chunk):
        n = min(chunk, n_streams - s0)
        s = (torch.arange(n, dtype=torch.int64, device=device) + (first_stream + s0))[:, None, None]
        x = (s << 24) ^ (f << 8) ^ k ^ i64(seed ^ (codec << 56))
        x = x + i64(0x9E3779B97F4A7C15)
        x = (x ^ lsr(x, 30)) * i64(0xBF58476D1CE4E5B9)
        x = (x ^ lsr(x, 27)) * i64(0x94D049BB133111EB)
        x = x ^ lsr(x, 31)
        b = ((x[..., None] >> sh) & 1).to(torch.uint8).reshape(n, n_frames, nw * 64)
        out[s0:s0 + n] = b[:, :, :fb]
    return out


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            with open(p) as f:
                d = json.load(f)
            if "hbm_gbs" in d:
                return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock / throttle-reason samples during the timed region: NVML (nvidia_ml_py, one sample every few ms) when it
    loads, else `nvidia-smi` polling."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.index = index
        self.rows = []      # (sm MHz, max MHz, watts, [active reason names])
        self.stop = threading.Event()
        self.th = None
        self.nvml = None
        self.handle = None
        self.source = "nvidia-smi"
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical devices: map the CUDA ordinal through CUDA_VISIBLE_DEVICES when it is a plain list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            phys = index
            if vis and all(x.strip().isdigit() for x in vis.split(",")):
                phys = int(vis.split(",")[index])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
            self.source = "nvml"
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n, h = self.nvml, self.handle
        sm = float(n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM))
        mx = float(n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM))
        pw = n.nvmlDeviceGetPowerUsage(h) / 1000.0
        try:
            bits = n.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
            bits = n.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        masks = [getattr(n, "nvmlClocksThrottleReasonHwSlowdown", 0x8), getattr(n, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 getattr(n, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20), getattr(n, "nvmlClocksThrottleReasonSwPowerCap", 0x4)]
        self.rows.append((sm, mx, pw, [nm for nm, m in zip(self.NAMES, masks) if bits & m]))

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
        parts = [x.strip() for x in out.strip().split(",")]
        if len(parts) >= 7:
            self.rows.append((float(parts[0]), float(parts[1]), float(parts[2]),
                              [nm for k, nm in enumerate(self.NAMES) if parts[3 + k].lower().startswith("active")]))

    def _run(self):
        while not self.stop.is_set():
            try:
                if self.nvml:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            self.stop.wait(0.004 if self.nvml else 0.1)

    def __enter__(self):
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": self.source}
        sm = sorted(r[0] for r in self.rows)
        reasons = [nm for nm in self.NAMES if any(nm in r[3] for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(r[1] for r in self.rows), "reasons": reasons,
                "power_w": round(max(r[2] for r in self.rows), 1), "samples": len(self.rows), "source": self.source}


def bind_to_gpu_numa_node(local_rank):
    """Run this rank (and first-touch its pinned host buffers) on the CPUs next to its GPU: with eight ranks gathering
    PCM at once the host side is the limit (DESIGN.md section 6), and remote-node staging makes it worse.  Returns a short
    description; does nothing when the box exposes no NUMA topology."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local_rank)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        base = "/sys/bus/pci/devices/" + bdf
        node = int(open(base + "/numa_node").read().strip())
        if node < 0:
            return "numa: none exposed (%s)" % bdf
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return "numa: node %d has no allowed cpu" % node
        os.sched_setaffinity(0, cpus)
        return "numa: node %d, %d cpus (%s)" % (node, len(cpus), bdf)
    except Exception as e:
        return "numa: not bound (%s)" % type(e).__name__


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def channel_like_frames(codec, n_streams, n_frames, seed):
    """BASELINE.json configs[4]-shaped soft input: valid encoded frames, every channel bit flipped with p = 0.10, reliability 255 for unflipped and U[0,64) for flipped
    bits.  Returns uint8 [streams][frames][bits][2]."""
    import mbe_testlib as T
    rng = np.random.default_rng(seed)
    enc7100 = getattr(T, "encode_imbe7100_frame", None)
    if codec == 1 and enc7100 is None:
        hard = T.random_hard_frames(codec, n_streams, n_frames, 0x7100)
    else:
        enc = T.encode_imbe7200_frame if codec == 0 else (enc7100 if codec == 1 else T.encode_ambe_frame)
        hard = np.zeros((n_streams, n_frames, FRAME_BITS[codec]), np.uint8)
        for b in range(n_streams):
            for f in range(n_frames):
                pb = rng.integers(0, 2, size=T.PARAM_BITS[codec], dtype=np.uint8)
                pb[0] = 0
                hard[b, f] = enc(pb).reshape(-1)
    return T.soften(hard, rng, flip_p=0.10)


def tone_unvoiced_frames(n_streams, n_frames, seed):
    """BASELINE.json configs[3]-shaped input (AMBE 3600x2400 only): frames built from parameter bits - a third tone / silence
    frames, a third unvoiced-only voice frames (FFT / WOLA / noise-generator path), a third ordinary voice frames - Golay
    encoded and PN scrambled into valid channel frames.  Returns uint8 [streams][frames][96]."""
    import mbe_testlib as T
    rng = np.random.default_rng(seed)
    frames = np.zeros((n_streams, n_frames, 96), np.uint8)
    for s in range(n_streams):
        for f in range(n_frames):
            p = rng.integers(0, 2, size=49, dtype=np.uint8)
            if (s + f // 5) % 3 == 0:
                p[0:6] = 1
            elif s % 2:
                p[38:42] = 0
            frames[s, f] = T.encode_ambe_frame(p).reshape(-1)
    return frames


def part_frames_numpy(codec, kind, first_stream, n_streams, n_frames):
    """Host copy of a part's input for global streams [first, first + n): the counter-based bits for "hard", 128 distinct
    seeded streams tiled over the range otherwise (the same 128 on every rank and on both arms)."""
    if kind == "hard":
        return counter_bits_numpy(codec, first_stream, n_streams, n_frames)
    B = 128
    base = tone_unvoiced_frames(B, n_frames, 0x2400) if kind == "tones" else (
        channel_like_frames(codec, B, n_frames, 0x50F7) if kind == "softch" else None)
    if base is None:  # "soft": random bits with random reliabilities
        rng = np.random.default_rng(0x2450)
        bits = counter_bits_numpy(codec, first_stream, n_streams, n_frames)
        return np.stack([bits, rng.integers(0, 256, size=bits.shape, dtype=np.uint8)], axis=-1)
    idx = (np.arange(n_streams) + first_stream) % B
    return np.ascontiguousarray(base[idx])


def load_cpu_reference():
    import mbe_testlib as T
    if T.ref_available(fast=True):
        return T.load_ref(fast=True).ref_bench_run, "reference", \
            "oracle/_ref/libmberef_fast.so (unmodified reference, dev-release flags: SIMD + fast-math + LTO)"
    if T.ref_available(fast=False):
        return T.load_ref(fast=False).ref_bench_run, "reference", "oracle/_ref/libmberef.so (unmodified reference, Release flags)"
    return T.load_oracle().mbo_run, "port", "oracle/libmbe_oracle.so (C restatement)"


def run_cpu_reference(parts, n_frames, steps, warmup, streams_per_thread):
    """Times the reference's CPU implementation (oracle/_ref dev-release build; the oracle port if the compiled reference is
    missing) on all host cores, worker threads pinned 1:1 to cores, on a bounded sample of the workload: global streams
    0 .. S-1 of every part with the same input bits the GPU arm decodes.  Returns (frames/s, info dict, seconds per step)."""
    import mbe_testlib as T
    cores = host_cores()
    fn, kind, flavour = load_cpu_reference()
    total_frames, total_sec, notes = 0, 0.0, []
    for codec, ikind in parts:
        soft = ikind in ("soft", "softch")
        spt = max(1, streams_per_thread // 50) if soft else streams_per_thread  # the reference's soft ECC is ~1 ms per IMBE frame
        S = min(cores * spt, 65536)
        frames = part_frames_numpy(codec, ikind, 0, S, n_frames)
        seeds = T.stream_seeds(S)
        pcm = np.zeros((S, n_frames, 160), np.int16)
        res = np.zeros((S, n_frames, 6), np.int32)
        times = []
        for it in range(warmup + steps):
            sec = fn(codec, int(soft), S, n_frames, T._ptr(frames), T._ptr(seeds), T._ptr(pcm), None, T._ptr(res), None, None, cores)
            if it >= warmup:
                times.append(sec)
        total_sec += float(np.mean(times))
        total_frames += S * n_frames
        notes.append("%s %s: %d streams x %d frames (%d per thread)" % (CODEC_NAMES[codec], ikind, S, n_frames, spt))
    fps = total_frames / total_sec
    info = {"value": fps, "unit": "frames/s", "cores": cores, "kind": kind,
            "sample": "%s per step; one stream per task over %d pthreads pinned 1:1 to cores; %s; input = the GPU arm's bits "
                      "for global streams 0.. of each part" % ("; ".join(notes), cores, flavour),
            "cpu_model": cpu_model(), "frames_per_s_per_core": fps / cores}
    return fps, info, total_sec


def dump_outputs(out_dir, parts, bounds, first_global, n_frames, outs):
    """Writes the --dump-outputs sample (see the module docstring) of the device outputs `outs` [(pcm, results)] per part."""
    per_stream = n_frames * 160 * 4 + n_frames * 6 * 8 + 8
    header = 4096                                     # bound on one .npy header (np.save pads it to 128 bytes here)
    k_max = min(DUMP_MAX_STREAMS, (DUMP_BUDGET_BYTES - 3 * len(parts) * header) // (per_stream * len(parts)))
    if k_max < 1:
        raise SystemExit("bench.py: --dump-outputs: one stream of %d frames per part exceeds %d bytes" % (n_frames, DUMP_BUDGET_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for p, (codec, kind) in enumerate(parts):
        n = bounds[p + 1] - bounds[p]
        idx = np.sort(np.random.default_rng(DUMP_SEED + p).choice(n, size=min(n, k_max), replace=False))
        pcm = outs[p][0][idx].cpu().numpy().astype(np.float32)
        res = outs[p][1][idx].cpu().numpy().astype(np.int64)
        res[..., 5] &= 0xffffffff                     # flags are uint32
        name = os.path.join(out_dir, "%s_%s_" % (CODEC_NAMES[codec], kind))
        np.save(name + "streams.npy", (idx + first_global + bounds[p]).astype(np.float64))
        np.save(name + "pcm.npy", pcm)
        np.save(name + "results.npy", res.astype(np.float64))


def build_workload(args, world):
    """-> dict(parts=[(codec id, input kind)], total streams (None: per-GPU count), per_gpu, scaling, what)."""
    custom = args.codec is not None or args.soft or args.soft_channel or args.tones_unvoiced
    if custom:
        codec = "ambe3600x2400" if args.tones_unvoiced else (args.codec or "ambe3600x2450")
        kind = "tones" if args.tones_unvoiced else ("softch" if args.soft_channel else ("soft" if args.soft else "hard"))
        per_gpu = args.streams or 65536
        return {"parts": [(CODEC_IDS[codec], kind)], "total": per_gpu * world, "scaling": "weak", "config": None,
                "what": "custom: %s %s input, %d streams per GPU" % (codec, kind, per_gpu)}
    c = CONFIGS[args.config]
    parts = [(CODEC_IDS[n], k) for n, k in c["parts"]]
    if c["scaling"] == "weak":
        per_gpu = args.streams or c["streams"]
        return {"parts": parts, "total": per_gpu * world, "scaling": "weak", "config": args.config, "what": c["what"]}
    return {"parts": parts, "total": args.streams or c["streams"], "scaling": "strong", "config": args.config, "what": c["what"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 3, 4], help="BASELINE.json configs[N] (default 2: the headline)")
    ap.add_argument("--codec", default=None, choices=list(CODEC_NAMES.values()), help="custom single-codec workload")
    ap.add_argument("--streams", type=int, default=None,
                    help="total streams (sharded configs 2-4) or streams per GPU (config 1 and custom workloads)")
    ap.add_argument("--frames", type=int, default=50, help="frames per stream per step")
    ap.add_argument("--soft", action="store_true", help="custom: soft-decision input (bit + reliability per channel bit), random reliabilities")
    ap.add_argument("--soft-channel", action="store_true",
                    help="custom: soft-decision input shaped like BASELINE.json configs[4]: valid encoded frames, every channel bit "
                         "flipped with p = 0.10, reliability 255 for unflipped and U[0,64) for flipped bits (128 distinct "
                         "streams tiled over the batch)")
    ap.add_argument("--tones-unvoiced", action="store_true",
                    help="custom: BASELINE.json configs[3]-shaped input (forces --codec ambe3600x2400): tone, unvoiced-only and voice "
                         "frames from parameter bits, valid channel frames (128 distinct streams tiled over the batch)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a seeded sample of the last timed step's PCM and results to DIR/*.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    F = args.frames
    wl = build_workload(args, world)
    parts = wl["parts"]
    total_streams = wl["total"]

    sys.path.insert(0, os.path.join(ROOT, "mbelib-neo_b200"))
    import importlib.util
    spec = importlib.util.spec_from_file_location("mbe_b200_sharding", os.path.join(ROOT, "mbelib-neo_b200", "sharding.py"))
    sharding = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(sharding)
    first_global, S = sharding.shard_range(total_streams, rank, world)     # this rank's block of global stream ids
    # the rank's streams are cut into one contiguous range per part (configs[4]: a third per codec)
    bounds = [S * i // len(parts) for i in range(len(parts) + 1)]
    bytes_in_per_frame = [FRAME_BITS[c] * (2 if k in ("soft", "softch") else 1) for c, k in parts]
    io_mb = sum((bounds[i + 1] - bounds[i]) * F * (bytes_in_per_frame[i] + 344) for i in range(len(parts))) / 1e6
    config = {"workload": wl["what"] + ", %d synthetic frames per stream per step" % F,
              "baseline_config": ("configs[%d]" % wl["config"]) if wl["config"] else None,
              "parts": ["%s/%s" % (CODEC_NAMES[c], k) for c, k in parts],
              "total_streams": total_streams, "streams_this_rank": S, "frames_per_stream": F,
              "sharding": "contiguous global stream ids, %d per rank over %d rank(s), no collective" % (S, world),
              "input": "counter-based splitmix64 bits keyed on (codec, global stream, frame): identical on every arm"
                       if all(k == "hard" for _, k in parts) else "128 seeded distinct streams tiled over the batch",
              "l2": "inputs+outputs per step on this rank (%.0f MB) exceed the 126 MB L2" % io_mb}

    if args.impl == "reference":
        if rank != 0:
            return 0
        warm = max(1, min(args.warmup, 3))
        fps, info, sec = run_cpu_reference(parts, F, args.steps, warm, streams_per_thread=1000)
        line = {"impl": "reference", "metric": "decoded frames/sec", "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": warm, "ms_per_step": sec * 1e3, "higher_is_better": True,
                "scaling": wl["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "realtime_channels": fps / 50.0, "cpu_baseline": info,
                "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist
    from __graft_entry__ import load_package
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the product has no CPU path (use --impl reference for the CPU arm)")
    pkg = load_package()
    torch.cuda.set_device(local_rank)
    numa_note = bind_to_gpu_numa_node(local_rank) if world > 1 else "numa: single rank, not bound"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)

    dec = pkg.Decoder(max_streams=max(S, 1), device=local_rank)
    dec.init_streams(0, S, sharding.stream_seeds(first_global, S))

    # ---- inputs, one tensor per part: rot[p] is a list of frame sets the steps rotate through
    gen = torch.Generator(device=dev)
    gen.manual_seed(0x2450 + rank)
    rot, outs = [], []
    for p, (codec, kind) in enumerate(parts):
        s0, n = bounds[p], bounds[p + 1] - bounds[p]
        fb = FRAME_BITS[codec]
        if kind == "hard":
            x = counter_bits_torch(codec, first_global + s0, n, F, dev)
        elif kind == "soft":
            x = torch.stack((counter_bits_torch(codec, first_global + s0, n, F, dev),
                             torch.randint(0, 256, (n, F, fb), dtype=torch.uint8, device=dev, generator=gen)), dim=-1).contiguous()
        else:
            B = 128
            base = torch.from_numpy(part_frames_numpy(codec, kind, 0, B, F)).to(dev)
            idx = (torch.arange(n, device=dev) + (first_global + s0)) % B
            x = base[idx].contiguous()
        sets = [x]
        # Short launches (a real-time server decodes ONE 20 ms frame per stream per launch) must not see the same frames
        # launch after launch: a stream fed the same frame twice has a perfectly stable pitch, which sends every low harmonic
        # through the phase-interpolated (one cosf per sample) path and times a workload nobody has.  Rotate through enough
        # different frame sets to cover 50 frames per stream.
        if F < 50 and kind in ("hard", "soft"):
            for k in range(1, min(50 // F, 25)):
                y = torch.randint(0, 2, (n, F, fb), dtype=torch.uint8, device=dev, generator=gen)
                if kind == "soft":
                    y = torch.stack((y, torch.randint(0, 256, (n, F, fb), dtype=torch.uint8, device=dev, generator=gen)), dim=-1).contiguous()
                sets.append(y)
        rot.append(sets)
        outs.append((torch.empty((n, F, 160), dtype=torch.int16, device=dev), torch.empty((n, F, 6), dtype=torch.int32, device=dev)))
    stream = torch.cuda.Stream(device=dev)
    step_no = [0]

    def step_dev():
        for p, (codec, kind) in enumerate(parts):
            n = bounds[p + 1] - bounds[p]
            if n == 0:
                continue
            fr = rot[p][step_no[0] % len(rot[p])]
            dec.process_frames_dev(codec, 1 if kind in ("soft", "softch") else 0, bounds[p], n, F, fr.data_ptr(),
                                   outs[p][0].data_ptr(), 0, outs[p][1].data_ptr(), 0, stream.cuda_stream)
        step_no[0] += 1

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        return sharding.max_over_ranks(x, device=dev)

    # ---- device-resident arm ----
    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            step_dev()
    barrier()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    dec.set_kernel_timing(True)     # an event pair around every kernel launch, on the stream it runs on (kernel_timing below)
    l0 = dec.launches
    with ClockSampler(local_rank) as clk:
        barrier()
        with torch.cuda.stream(stream):
            evs[0].record(stream)
            for k in range(args.steps):
                step_dev()
                evs[k + 1].record(stream)
        stream.synchronize()
        barrier()
    launches = dec.launches - l0
    kernel_ms, bank_work = dec.kernel_timing()
    dec.set_kernel_timing(False)
    kernel_path = dec.kernel_path()
    total_ms = max_over_ranks(evs[0].elapsed_time(evs[-1]))
    per_step_ms = [evs[k].elapsed_time(evs[k + 1]) for k in range(args.steps)]
    kern_ms = float(np.mean(per_step_ms))
    value = total_streams * F * args.steps / (total_ms * 1e-3)
    clocks = clk.summary()

    # sanity: the PCM that came out is not silence and statuses are valid
    for p in range(len(parts)):
        if bounds[p + 1] - bounds[p] == 0:
            continue
        chk = outs[p][0][:64].abs().max().item()
        st_min = int(outs[p][1][:, :, 0].min().item())
        if (chk == 0 or st_min < 0) and not os.environ.get("MBE_B200_SKIP_KERNELS"):   # (timing experiments skip kernels)
            raise SystemExit("bench.py: device path produced silence or error statuses (part %d: max |pcm| %d, min status %d)" % (p, chk, st_min))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, parts, bounds, first_global, F, outs)

    # ---- end-to-end arm: host frames in, host PCM + results out, through the host-pointer C-ABI calls ----
    e2e = None
    if not args.no_e2e and S > 0:
        import ctypes
        lib, h = dec.lib, dec.h
        vp = ctypes.c_void_p
        host = []   # per part: (list of pinned frame sets, packed frames or None, pcm, results)
        h2d = d2h = h2d_packed = 0
        all_hard = all(k == "hard" for _, k in parts) and all(len(r) == 1 for r in rot)
        for p, (codec, kind) in enumerate(parts):
            n = bounds[p + 1] - bounds[p]
            sets = []
            for x in rot[p]:
                hx = torch.empty(tuple(x.shape), dtype=torch.uint8, pin_memory=True)
                hx.copy_(x)
                sets.append(hx.numpy())
            packed = None
            if all_hard:
                packed = torch.from_numpy(pkg.pack_frames(codec, sets[0])).pin_memory().numpy()
                h2d_packed += packed.size
            h_pcm = torch.empty((n, F, 160), dtype=torch.int16, pin_memory=True).numpy()
            h_res = torch.empty((n, F, 6), dtype=torch.int32, pin_memory=True).numpy()
            host.append((sets, packed, h_pcm, h_res))
            h2d += sets[0].size
            d2h += n * F * (320 + RESULT_BYTES)
        host_step = [0]

        def step_host(use_packed):
            for p, (codec, kind) in enumerate(parts):
                n = bounds[p + 1] - bounds[p]
                if n == 0:
                    continue
                sets, packed, h_pcm, h_res = host[p]
                if use_packed:
                    rc = lib.mbe_b200_process_frames_packed(h, codec, bounds[p], n, F, packed.ctypes.data_as(vp), h_pcm.ctypes.data_as(vp),
                                                            None, h_res.ctypes.data_as(vp), None)
                else:
                    cur = sets[host_step[0] % len(sets)]
                    rc = lib.mbe_b200_process_frames(h, codec, 1 if kind in ("soft", "softch") else 0, bounds[p], n, F,
                                                     cur.ctypes.data_as(vp), h_pcm.ctypes.data_as(vp), None, h_res.ctypes.data_as(vp), None)
                if rc != 0:
                    raise SystemExit("mbe_b200_process_frames failed: %s" % lib.mbe_b200_last_error(h).decode())
            host_step[0] += 1

        def time_host(use_packed):
            for _ in range(max(1, min(args.warmup, 2))):
                step_host(use_packed)
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                step_host(use_packed)          # returns when PCM + results are in host memory
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            sec = max_over_ranks(t1 - t0)
            barrier()
            return sec

        sec_bytes = time_host(False)
        if float(np.abs(host[0][2][:64]).max()) == 0:
            raise SystemExit("bench.py: e2e path produced silence")
        res_bytes = {"value": total_streams * F * args.steps / sec_bytes, "unit": "frames/s", "h2d_bytes_per_step": int(h2d),
                     "ms_per_step": sec_bytes * 1e3 / args.steps,
                     "note": "mbe_b200_process_frames: one byte per channel bit (the reference's char fr[][] layout)"}
        res_packed = None
        if all_hard:
            sec_packed = time_host(True)
            res_packed = {"value": total_streams * F * args.steps / sec_packed, "unit": "frames/s", "h2d_bytes_per_step": int(h2d_packed),
                          "ms_per_step": sec_packed * 1e3 / args.steps,
                          "note": "mbe_b200_process_frames_packed: hard bits packed eight per byte (SURVEY 8(f)-1)"}
        # what the host links allow: the step's bytes moved by plain copies on two streams, every rank at once
        s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

        def link_time(packed_in):
            srcs = [torch.from_numpy(hp[1] if packed_in else hp[0][0]) for hp in host]
            dsts = [torch.empty(x.shape, dtype=torch.uint8, device=dev) for x in srcs]
            back = [(torch.from_numpy(hp[2]), torch.from_numpy(hp[3])) for hp in host]
            best = None
            for it in range(3):
                barrier()
                t0 = time.perf_counter()
                with torch.cuda.stream(s_in):
                    for a, b in zip(srcs, dsts):
                        b.copy_(a, non_blocking=True)
                with torch.cuda.stream(s_out):
                    for p in range(len(parts)):
                        back[p][0].copy_(outs[p][0], non_blocking=True)
                        back[p][1].copy_(outs[p][1], non_blocking=True)
                torch.cuda.synchronize()
                t = max_over_ranks(time.perf_counter() - t0)
                best = t if best is None else min(best, t)
            del dsts
            return best

        use_packed_headline = world > 1 and res_packed is not None
        head = res_packed if use_packed_headline else res_bytes
        t_link = link_time(use_packed_headline)
        link_fps = total_streams * F / t_link
        e2e = {"value": head["value"], "unit": "frames/s", "h2d_bytes_per_step": head["h2d_bytes_per_step"],
               "d2h_bytes_per_step": int(d2h), "ms_per_step": head["ms_per_step"],
               "input": "bit-packed channel frames" if use_packed_headline else "one byte per channel bit",
               "bytes_input": res_bytes, "packed_input": res_packed, "host_binding": numa_note,
               "link_ceiling": {"value": link_fps, "unit": "frames/s", "ms_per_step": t_link * 1e3,
                                "gbytes_per_s_this_rank": (head["h2d_bytes_per_step"] + d2h) / t_link / 1e9,
                                "note": "the step's host<->device bytes as plain pinned copies (in and out on two streams), all ranks "
                                        "at once, best of 3, max over ranks: no kernel, no pipeline"},
               "frac_of_link": head["value"] / link_fps,
               "frac_of_device": head["value"] / value,
               "note": "pinned host frame bits in, int16 PCM + results to pinned host memory, wall clock around the blocking "
                       "C-ABI calls, max over ranks; packed input is the headline at N > 1 (the host links are the limit there)"}

    # ---- rooflines ----
    # `roofline` is the dominant kernel's: on the multi-kernel path the bank kernel (mbe_split_bank_kernel), whose launches were
    # bracketed by CUDA events on their own streams during the timed region and whose work (oscillator slots x 160 samples,
    # interpolated harmonics) the kernel counted itself; on the fused path the stream kernel.  `roofline_step` is the whole
    # step (every kernel) against the same FP32-issue peak, `roofline_hbm` the HBM view of the step.
    hbm_peak, peak_src = measured_peaks()
    consts = ncu_constants()
    alg_bytes = flops = dram = winstr = 0.0
    have_all = True
    per_part = []
    for p, (codec, kind) in enumerate(parts):
        n = bounds[p + 1] - bounds[p]
        alg_bytes += n * F * (bytes_in_per_frame[p] + 320 + RESULT_BYTES) + 2 * n * STATE_BYTES
        flops += n * F * FLOP_PER_FRAME[codec]
        c = consts.get("%s/%s" % (CODEC_NAMES[codec], kind))
        if c:
            dram += n * F * c["dram_bytes_per_frame"]
            winstr += n * F * c["warp_instr_per_frame"]
            per_part.append({"part": "%s/%s" % (CODEC_NAMES[codec], kind), **c})
        else:
            have_all = False
    sm_mhz = clocks.get("sm_mhz") or 1965.0
    fp32_issue_peak = 148 * 128 * sm_mhz * 1e6 / 1e12  # TFLOP/s, one non-fused op per lane per clock
    peak_note = ("148 SM x 128 FP32 lanes x %.0f MHz sampled SM clock, non-fused (mul and add issue separately because parity "
                 "forbids FMA contraction); the FMA-counted peak is 2x; the path has no dense contraction, so neither HBM nor "
                 "the tensor cores bound it (see roofline_hbm)" % sm_mhz)
    fp32_ach = flops / (kern_ms * 1e-3) / 1e12
    hbm_ach = alg_bytes / (kern_ms * 1e-3) / 1e9
    roofline_step = {"bound": "fp32-issue", "achieved": fp32_ach, "peak": fp32_issue_peak, "unit": "TFLOP/s",
                     "frac": fp32_ach / fp32_issue_peak, "step_ms": kern_ms, "algorithmic_flop_per_step": flops,
                     "flop_per_frame": {CODEC_NAMES[c]: FLOP_PER_FRAME[c] for c, _ in parts},
                     "note": "every kernel of the step: SURVEY 8(d)'s analytic FLOP per frame x frames / event-timed step"}
    kinds_ms = {k: v[0] for k, v in kernel_ms.items()}
    kinds_n = {k: v[1] for k, v in kernel_ms.items()}
    busy = sum(kinds_ms.values()) or 1.0
    kernels = {k: {"launches": kinds_n[k], "ms_total": kinds_ms[k], "ms_per_launch": kinds_ms[k] / max(1, kinds_n[k]),
                   "share_of_kernel_time": kinds_ms[k] / busy} for k in kinds_ms if kinds_n[k]}
    if kernel_path == 1 and kinds_n.get("bank"):
        # per slot: 160 x (6 rotation + 2 gain / window + 1 ordered add) = 1440 FLOP; per interpolated harmonic 160 x 46
        win_slots = bank_work["slots"] - bank_work["interpolated"]
        bank_flop = 1440.0 * win_slots + 160.0 * 46.0 * bank_work["interpolated"]
        # The step's kernels run on several streams at once, so an event pair around one launch also counts the time its
        # neighbours held the SMs: the sum of all bracketed durations is `concurrency` x the step.  The bank kernel's own
        # share of the step is its share of that sum; achieved = its FLOP / (step time x share).
        wall_ms = evs[0].elapsed_time(evs[-1])
        concurrency = busy / wall_ms
        share = kernels["bank"]["share_of_kernel_time"]
        ach = bank_flop / (wall_ms * share * 1e-3) / 1e12
        roofline = {"bound": "fp32-issue", "achieved": ach, "peak": fp32_issue_peak, "unit": "TFLOP/s", "frac": ach / fp32_issue_peak,
                    "traffic": None, "kernel": "mbe_split_bank_kernel",
                    "launch_ms": kernels["bank"]["ms_per_launch"] / concurrency, "launch_ms_bracketed": kernels["bank"]["ms_per_launch"],
                    "concurrency": concurrency, "launches": kinds_n["bank"],
                    "algorithmic_flop_per_launch": bank_flop / kinds_n["bank"],
                    "work": {"oscillator_slots": bank_work["slots"], "interpolated_harmonics": bank_work["interpolated"],
                             "frames_synthesised": bank_work["frames"],
                             "slots_per_frame": bank_work["slots"] / max(1, bank_work["frames"])},
                    "share_of_step": share,
                    "peak_source": peak_note,
                    "note": "launch durations are CUDA-event pairs on the launching streams inside the timed region; launch_ms = "
                            "bracketed duration / concurrency (see bench.py); the solo, cold-cache durations and the pipe "
                            "utilisation of the same launches are in profiles/ (ncu launch list, ncu_constants.json)"}
    else:
        roofline = dict(roofline_step)
        roofline.update({"traffic": None, "kernel": "mbe_stream_kernel", "launch_ms": kern_ms,
                         "algorithmic_flop_per_launch": flops, "peak_source": peak_note})
    if have_all and dram:
        roofline["traffic"] = dram
        roofline["traffic_source"] = ("ncu dram__bytes_read.sum + dram__bytes_write.sum per frame, all kernels of the path, x frames per "
                                      "step (profiles/ncu_constants.json)")
    if have_all and winstr:
        issue_peak = 148 * 4 * sm_mhz * 1e6   # warp-instructions per second, one per scheduler per clock
        issue_ach = winstr / (kern_ms * 1e-3)
        roofline["issue_slots"] = {"achieved": issue_ach / 1e9, "peak": issue_peak / 1e9, "unit": "G warp-instr/s",
                                   "frac": issue_ach / issue_peak, "warp_instr_per_frame": winstr / (S * F),
                                   "source": "ncu smsp__inst_executed.sum per frame, all kernels of the path "
                                             "(profiles/ncu_constants.json) x frames per step / event-timed step"}
        roofline["ncu"] = per_part
    roofline_hbm = {"bound": "hbm", "achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_ach / hbm_peak,
                    "traffic": dram if (have_all and dram) else None, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": alg_bytes,
                    "note": "bit-in / PCM-out / state traffic of the step: ~1 KB per frame (the multi-kernel path adds its "
                            "descriptors, ~3 KB per frame written and read once: see traffic); HBM stays > 90 % idle"}
    line = {"metric": "decoded frames/sec", "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": wl["scaling"],
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "realtime_channels": value / 50.0, "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
            "roofline": roofline, "roofline_step": roofline_step, "roofline_hbm": roofline_hbm,
            "kernel_path": "multi-kernel (parameter + bank + unvoiced)" if kernel_path == 1 else "fused", "kernels": kernels}

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        _, info, _ = run_cpu_reference(parts, F, 2, 1, streams_per_thread=1000)
        line["cpu_baseline"] = info
    dec.close()
    if world > 1:
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(line))
    return 0


if __name__ == "__main__":
    sys.exit(main())
