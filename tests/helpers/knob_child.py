"""Child process of the knob tests: libmbe_b200 reads its tuning knobs (MBE_B200_*) from the environment once per process,
so a test that varies them runs the library here, under the environment its parent chose.

    knob_child.py plan N [N ...]     prints {N: mbe_b200_pipeline_plan(N)} as JSON (no device needed)
    knob_child.py run IN.npz OUT.npz  decodes the inputs of tests/test_gpu_knobs.py through every host-side path on
                                      cuda:0 and saves every output, the end states and the launch count of each call

The child only runs the library and records what it returns; the parent checks it against the CPU oracle.
"""
import ctypes
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from __graft_entry__ import load_package  # noqa: E402


def plan(ns):
    lib = load_package().load_library()
    buf = (ctypes.c_int * 64)()
    out = {}
    for n in ns:
        k = lib.mbe_b200_pipeline_plan(int(n), buf, 64)
        assert 0 <= k <= 64, (n, k)
        out[int(n)] = list(buf[:k])
    print(json.dumps(out))


def run(inp, outp):
    import torch
    pkg = load_package()
    z = dict(np.load(inp))
    M, f0 = int(z["max_streams"]), int(z["first_stream"])
    seeds = z["seeds"]
    cuts = {k: [(int(a), int(b)) for a, b in z[k]] for k in ("cuts3", "cuts0")}
    dev = torch.device("cuda", 0)
    dec = pkg.Decoder(max_streams=M, device=0)
    res_i32 = lambda r: np.ascontiguousarray(r).view(np.int32).reshape(r.shape[0], r.shape[1], 6)
    out, calls = {}, []

    def counted(row, n, a, b, kind, pipelined, indexed, fn):
        n0 = dec.launches
        r = fn()
        calls.append(dict(row=row, n=n, frames=b - a, kind=kind, pipelined=pipelined, indexed=indexed,
                          launches=dec.launches - n0))
        return r

    def keep(row, parts, state, rng, fields=("pcm", "pcmf", "results", "bits")):
        for k in fields:
            x = np.concatenate([p[k] for p in parts], axis=1)
            out[row + "." + k] = res_i32(x) if k == "results" and x.dtype == pkg.RESULT_DTYPE else x
        out[row + ".state"], out[row + ".rng"] = state, rng

    def sentinel(n, F, codec, bits=True):
        d = dict(pcm=torch.full((n, F, 160), 0x5555, dtype=torch.int16, device=dev),
                 pcmf=torch.full((n, F, 160), 1.5, dtype=torch.float32, device=dev),
                 results=torch.full((n, F, 6), 77, dtype=torch.int32, device=dev))
        if bits:
            d["bits"] = torch.full((n, F, pkg.PARAM_BITS[codec]), 9, dtype=torch.uint8, device=dev)
        return d

    def to_host(d):
        return {k: v.cpu().numpy() for k, v in d.items()}

    def init():
        dec.init_streams(0, M, seeds)

    # contiguous calls: streams [f0, f0 + n) of the pool, every row in two calls of different lengths
    for row, codec, soft, key, row_cuts in (("host3", 3, 0, "frames3", cuts["cuts3"]), ("host0", 0, 0, "frames0", cuts["cuts0"]),
                                            ("soft0", 0, 1, "soft0", cuts["cuts0"])):
        fr = z[key]
        n = fr.shape[0]
        init()
        parts = [counted(row, n, a, b, int(soft), True, False,
                         lambda: dec.process_frames(codec, np.ascontiguousarray(fr[:, a:b]), soft=bool(soft), first_stream=f0,
                                                    want_float=True)) for a, b in row_cuts]
        keep(row, parts, dec.export_state(f0, n), dec.export_rng(f0, n))

    fr3, cuts3 = z["frames3"], cuts["cuts3"]
    n3 = fr3.shape[0]

    # device-resident call on the context's own stream (forks its stream ranges over the internal streams)
    init()
    parts = []
    for a, b in cuts3:
        x = torch.from_numpy(np.ascontiguousarray(fr3[:, a:b])).to(dev)
        o = sentinel(n3, b - a, 3)
        torch.cuda.synchronize()
        counted("dev3", n3, a, b, 0, False, False,
                lambda: dec.process_frames_dev(3, 0, f0, n3, b - a, x.data_ptr(), o["pcm"].data_ptr(), o["pcmf"].data_ptr(),
                                               o["results"].data_ptr(), o["bits"].data_ptr(), cuda_stream=0))
        dec.synchronize()
        parts.append(to_host(o))
    keep("dev3", parts, dec.export_state(f0, n3), dec.export_rng(f0, n3))

    # the asynchronous half of the host path, into page-locked buffers
    init()
    parts = []
    for a, b in cuts3:
        x = np.ascontiguousarray(fr3[:, a:b])
        o = dict(pcm=pkg.host_alloc((n3, b - a, 160), np.int16), pcmf=pkg.host_alloc((n3, b - a, 160), np.float32),
                 results=pkg.host_alloc((n3, b - a), pkg.RESULT_DTYPE),
                 bits=pkg.host_alloc((n3, b - a, pkg.PARAM_BITS[3]), np.uint8))

        def submit_and_wait():
            dec.submit_frames(3, x, o, first_stream=f0)
            dec.wait()
        counted("submit3", n3, a, b, 0, True, False, submit_and_wait)
        parts.append({k: v.copy() for k, v in o.items()})
        for v in o.values():
            pkg.host_free(v)
    keep("submit3", parts, dec.export_state(f0, n3), dec.export_rng(f0, n3))

    # bit-packed input
    init()
    packed = pkg.pack_frames(3, fr3)
    parts = [counted("packed3", n3, a, b, 2, True, False,
                     lambda: dec.process_frames_packed(3, np.ascontiguousarray(packed[:, a:b]), first_stream=f0, want_float=True))
             for a, b in cuts3]
    keep("packed3", parts, dec.export_state(f0, n3), dec.export_rng(f0, n3))

    # indexed calls: element i is slot slots[i]; the accepted elements' slots start from row host3's seeds
    slots, ok, idle = z["slots"], z["accepted"], z["idle_slots"]
    for row in ("idx3", "idxdev3"):
        init()
        dec.init_streams_indexed(slots[ok], seeds[f0:f0 + n3][ok])
        out[row + ".idle_state_before"], out[row + ".idle_rng_before"] = dec.export_state_indexed(idle), dec.export_rng_indexed(idle)
        parts = []
        if row == "idxdev3":
            d_slots = torch.from_numpy(slots).to(dev)
            s = torch.cuda.Stream(device=dev)
        for a, b in cuts3:
            x = np.ascontiguousarray(fr3[:, a:b])
            if row == "idx3":
                parts.append(counted(row, n3, a, b, 0, True, True,
                                     lambda: dec.process_indexed(3, slots, x, input=pkg.INPUT_HARD, want_float=True)))
                continue
            xd = torch.from_numpy(x).to(dev)
            o = sentinel(n3, b - a, 3)
            torch.cuda.synchronize()
            with torch.cuda.stream(s):
                counted(row, n3, a, b, 0, False, True,
                        lambda: dec.process_indexed_dev(3, pkg.INPUT_HARD, d_slots.data_ptr(), n3, b - a, xd.data_ptr(),
                                                        o["pcm"].data_ptr(), o["pcmf"].data_ptr(), o["results"].data_ptr(),
                                                        o["bits"].data_ptr(), cuda_stream=s.cuda_stream))
            s.synchronize()
            parts.append(to_host(o))
        keep(row, parts, dec.export_state_indexed(slots[ok]), dec.export_rng_indexed(slots[ok]))
        out[row + ".idle_state_after"], out[row + ".idle_rng_after"] = dec.export_state_indexed(idle), dec.export_rng_indexed(idle)

    # parameter-bit input (mbe_process<Codec>Data): the bits and ECC results of row host3's frames
    bits, res = dec.decode_frames(3, fr3)
    bits = bits.reshape(n3, fr3.shape[1], -1)
    res = res.reshape(n3, fr3.shape[1])
    init()
    parts = [counted("data3", n3, a, b, 0, False, False,
                     lambda: dec.process_data(3, bits[:, a:b], results=res[:, a:b], first_stream=f0, want_float=True))
             for a, b in cuts3]
    keep("data3", parts, dec.export_state(f0, n3), dec.export_rng(f0, n3), fields=("pcm", "pcmf", "results"))
    init()
    parts = []
    s = torch.cuda.Stream(device=dev)
    for a, b in cuts3:
        xb = torch.from_numpy(np.ascontiguousarray(bits[:, a:b])).to(dev)
        o = sentinel(n3, b - a, 3, bits=False)
        o["results"] = torch.from_numpy(res_i32(res[:, a:b])).to(dev)       # in / out
        torch.cuda.synchronize()
        counted("datadev3", n3, a, b, 0, False, False,
                lambda: dec._check(dec.lib.mbe_b200_process_data_dev(dec.h, 3, f0, n3, b - a, xb.data_ptr(), o["results"].data_ptr(),
                                                                     o["pcm"].data_ptr(), o["pcmf"].data_ptr(), s.cuda_stream),
                                   "process_data_dev"))
        s.synchronize()
        parts.append(to_host(o))
    keep("datadev3", parts, dec.export_state(f0, n3), dec.export_rng(f0, n3), fields=("pcm", "pcmf", "results"))

    buf = (ctypes.c_int * 64)()
    plans = {}
    for n in sorted({c["n"] for c in calls}):
        k = dec.lib.mbe_b200_pipeline_plan(n, buf, 64)
        plans[n] = list(buf[:k])
    meta = dict(calls=calls, plans=plans, kernel_path=dec.kernel_path(),
                sm_count=torch.cuda.get_device_properties(dev).multi_processor_count,
                env={k: v for k, v in os.environ.items() if k.startswith("MBE_B200_") and k != "MBE_B200_LIB"})
    dec.close()
    out["meta"] = np.array(json.dumps(meta))
    np.savez(outp, **out)
    for c in calls:
        print("%-9s n=%5d frames=%d launches=%d" % (c["row"], c["n"], c["frames"], c["launches"]))


if __name__ == "__main__":
    if sys.argv[1] == "plan":
        plan(sys.argv[2:])
    else:
        assert sys.argv[1] == "run"
        run(sys.argv[2], sys.argv[3])
