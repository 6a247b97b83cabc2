"""Child process of the indexed parameter-bit knob test (tests/test_gpu_data_indexed.py): libmbe_b200 reads its tuning
knobs (MBE_B200_*) from the environment once per process, so the test runs the library here under each setting.

    data_knob_child.py run IN.npz OUT.npz   decodes the parameter bits and decode contexts of IN.npz through every
                                            indexed parameter-bit path on cuda:0 (host one byte per bit, host packed,
                                            submit/wait, device-resident on a caller's stream) and saves every output,
                                            the end states and the launch count of each call

The child only runs the library and records what it returns; the parent checks it against the CPU oracle.
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from __graft_entry__ import load_package  # noqa: E402

ROWS = ("dataidx3", "dataidxpk3", "datasubmit3", "dataidxdev3")


def run(inp, outp):
    import torch
    pkg = load_package()
    z = dict(np.load(inp))
    M, f0 = int(z["max_streams"]), int(z["first_stream"])
    seeds, bits, res_in = z["seeds"], z["bits"], z["results"]
    slots, ok, idle = z["slots"], z["accepted"], z["idle_slots"]
    cuts = [(int(a), int(b)) for a, b in z["cuts"]]
    n, codec = bits.shape[0], 3
    packed = pkg.pack_params(codec, bits)
    res_dt = np.ascontiguousarray(res_in).view(pkg.RESULT_DTYPE).reshape(n, -1)
    dev = torch.device("cuda", 0)
    dec = pkg.Decoder(max_streams=M, device=0)
    res_i32 = lambda r: np.ascontiguousarray(r).view(np.int32).reshape(r.shape[0], r.shape[1], 6)
    out, calls = {}, []

    def counted(row, a, b, pipelined, fn):
        n0 = dec.launches
        r = fn()
        calls.append(dict(row=row, n=n, frames=b - a, kind=0, pipelined=pipelined, indexed=True,
                          launches=dec.launches - n0))
        return r

    for row in ROWS:
        dec.init_streams(0, M, seeds)
        dec.init_streams_indexed(slots[ok], seeds[f0:f0 + n][ok])
        out[row + ".idle_state_before"], out[row + ".idle_rng_before"] = dec.export_state_indexed(idle), dec.export_rng_indexed(idle)
        parts = []
        s = torch.cuda.Stream(device=dev)
        d_slots = torch.from_numpy(slots).to(dev)
        for a, b in cuts:
            x, xp, r = (np.ascontiguousarray(v[:, a:b]) for v in (bits, packed, res_dt))
            if row == "dataidx3":
                parts.append(counted(row, a, b, True, lambda: dec.process_data_indexed(codec, slots, x, results=r, want_float=True)))
            elif row == "dataidxpk3":
                parts.append(counted(row, a, b, True, lambda: dec.process_data_indexed(codec, slots, xp, results=r, packed=True,
                                                                                       want_float=True)))
            elif row == "datasubmit3":
                o = dict(pcm=pkg.host_alloc((n, b - a, 160), np.int16), pcmf=pkg.host_alloc((n, b - a, 160), np.float32),
                         results=pkg.host_alloc((n, b - a), pkg.RESULT_DTYPE))
                o["results"][:] = r

                def submit_and_wait():
                    dec.submit_data_indexed(codec, slots, xp, o, packed=True)
                    dec.wait()
                counted(row, a, b, True, submit_and_wait)
                parts.append({k: v.copy() for k, v in o.items()})
                for v in o.values():
                    pkg.host_free(v)
            else:
                xd = torch.from_numpy(x).to(dev)
                rd = torch.from_numpy(res_i32(r)).to(dev)
                o = dict(pcm=torch.full((n, b - a, 160), 0x5555, dtype=torch.int16, device=dev),
                         pcmf=torch.full((n, b - a, 160), 1.5, dtype=torch.float32, device=dev))
                torch.cuda.synchronize()
                with torch.cuda.stream(s):
                    counted(row, a, b, False,
                            lambda: dec.process_data_indexed_dev(codec, False, d_slots.data_ptr(), n, b - a, xd.data_ptr(),
                                                                 rd.data_ptr(), o["pcm"].data_ptr(), o["pcmf"].data_ptr(),
                                                                 cuda_stream=s.cuda_stream))
                s.synchronize()
                parts.append(dict(pcm=o["pcm"].cpu().numpy(), pcmf=o["pcmf"].cpu().numpy(),
                                  results=rd.cpu().numpy().view(pkg.RESULT_DTYPE).reshape(n, b - a)))
        for k in ("pcm", "pcmf", "results"):
            x = np.concatenate([p[k] for p in parts], axis=1)
            out[row + "." + k] = res_i32(x) if k == "results" else x
        out[row + ".state"], out[row + ".rng"] = dec.export_state_indexed(slots[ok]), dec.export_rng_indexed(slots[ok])
        out[row + ".idle_state_after"], out[row + ".idle_rng_after"] = dec.export_state_indexed(idle), dec.export_rng_indexed(idle)

    import ctypes
    buf = (ctypes.c_int * 64)()
    k = dec.lib.mbe_b200_pipeline_plan(n, buf, 64)
    meta = dict(calls=calls, plans={str(n): list(buf[:k])}, kernel_path=dec.kernel_path(), rows=list(ROWS),
                env={k: v for k, v in os.environ.items() if k.startswith("MBE_B200_") and k != "MBE_B200_LIB"})
    dec.close()
    out["meta"] = np.array(json.dumps(meta))
    np.savez(outp, **out)
    for c in calls:
        print("%-12s n=%5d frames=%d launches=%d" % (c["row"], c["n"], c["frames"], c["launches"]))


if __name__ == "__main__":
    assert sys.argv[1] == "run"
    run(sys.argv[2], sys.argv[3])
