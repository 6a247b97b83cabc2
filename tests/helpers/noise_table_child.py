"""Child process of tests/test_gpu_noise_table.py: libmbe_b200 reads MBE_B200_NOISE_TABLE once per process, so each setting
decodes here, under the environment its parent chose.

    noise_table_child.py IN.npz OUT.npz

IN holds cases "<name>.codec", ".frames", ".seeds" and optionally ".state" / ".rng" (states imported before the call).  Every
case decodes on cuda:0 on the multi-kernel path; OUT gets its pcm, pcmf, results, end state and the unvoiced kernel's
counters (noise spectra from the table, computed in the kernel).
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from __graft_entry__ import load_package  # noqa: E402


def main(inp, outp):
    pkg = load_package()
    z = dict(np.load(inp))
    names = sorted({k.split(".")[0] for k in z})
    out = {}
    for name in names:
        codec = int(z[name + ".codec"])
        frames, seeds = z[name + ".frames"], z[name + ".seeds"]
        S = frames.shape[0]
        dec = pkg.Decoder(max_streams=S, device=0)
        dec.set_kernel_path(1)
        dec.init_streams(0, S, seeds)
        if name + ".state" in z:
            dec.import_state(z[name + ".state"], 0)
            dec.import_rng(z[name + ".rng"], 0)
        dec.set_kernel_timing(True)
        got = dec.process_frames(codec, frames, want_float=True)
        out[name + ".counters"] = np.array(dec.noise_table_counters(), np.int64)
        dec.set_kernel_timing(False)
        out[name + ".pcm"] = got["pcm"]
        out[name + ".pcmf"] = got["pcmf"]
        out[name + ".results"] = np.ascontiguousarray(got["results"]).view(np.int32).reshape(S, frames.shape[1], 6)
        out[name + ".state"] = dec.export_state(0, S)
        dec.close()
    np.savez(outp, **out)


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
