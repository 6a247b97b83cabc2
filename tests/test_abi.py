"""C-ABI surface checks that need no GPU: libmbe_b200.so loads, exports every entry point include/mbe_b200.h
declares, reports the codec geometry, and refuses to create a context without a CUDA device (no CPU fallback)."""
import ctypes
import os
import re

import numpy as np
import pytest

from __graft_entry__ import ROOT, load_package


@pytest.fixture(scope="module")
def pkg():
    p = load_package()
    if not os.path.exists(p.LIB_PATH):
        import subprocess
        import sys
        subprocess.check_call([sys.executable, os.path.join(ROOT, "mbelib-neo_b200", "build.py")])
    return p


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "mbe_b200.h")).read()
    return sorted(set(re.findall(r"MBE_B200_API\s+[\w\s\*]+?\b(mbe_b200_\w+)\s*\(", text)))


def test_header_declares_the_expected_entry_points():
    names = declared_symbols()
    for must in ("mbe_b200_create", "mbe_b200_destroy", "mbe_b200_process_frames", "mbe_b200_process_frames_dev",
                 "mbe_b200_decode_frames", "mbe_b200_process_data", "mbe_b200_synthesize_speech", "mbe_b200_floattoshort",
                 "mbe_b200_init_streams", "mbe_b200_export_state", "mbe_b200_import_state"):
        assert must in names
    assert len(names) >= 20


def test_library_exports_every_declared_symbol(pkg):
    lib = pkg.load_library()
    for name in declared_symbols():
        assert hasattr(lib, name), "libmbe_b200.so does not export %s" % name
    assert set(pkg.exported_symbols()) == set(declared_symbols())


def test_geometry_and_version(pkg):
    lib = pkg.load_library()
    assert b"sm_100a" in lib.mbe_b200_version()
    fb, pb = ctypes.c_int(), ctypes.c_int()
    want = {0: (184, 88), 1: (168, 88), 2: (96, 49), 3: (96, 49)}
    for codec, (f, p) in want.items():
        assert lib.mbe_b200_geometry(codec, ctypes.byref(fb), ctypes.byref(pb)) == 0
        assert (fb.value, pb.value) == (f, p)
        assert pkg.FRAME_BITS[codec] == f and pkg.PARAM_BITS[codec] == p
    assert lib.mbe_b200_geometry(4, ctypes.byref(fb), ctypes.byref(pb)) == -1


def test_result_struct_layout_matches_header(pkg):
    assert pkg.RESULT_DTYPE.itemsize == 24
    assert pkg.RESULT_DTYPE.names == ("status", "c0_errors", "protected_errors", "c4_errors", "total_errors", "flags")
    assert pkg.PARMS_BYTES == 2604


def test_no_cpu_fallback(pkg):
    """Without a CUDA device the product must fail loudly, not decode on the CPU."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    with pytest.raises(pkg.MbeB200Error) as e:
        pkg.Decoder(max_streams=4, device=0)
    assert "no CUDA device" in str(e.value) or "-3" in str(e.value)


def test_product_does_not_link_the_oracle(pkg):
    """The product library has no dependency on oracle/ (the oracle is test infrastructure)."""
    out = os.popen("ldd %s" % pkg.LIB_PATH).read()
    assert "oracle" not in out and "mberef" not in out
    src = open(os.path.join(ROOT, "mbelib-neo_b200", "__init__.py")).read()
    assert "oracle" not in src.replace("no CPU fallback", "")


def test_pool_has_no_cpu_fallback(pkg):
    """mbe_b200_pool_create over "every visible device" fails with MBE_B200_E_NOGPU when there is none."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    assert pkg.load_library().mbe_b200_device_count() == 0
    with pytest.raises(pkg.MbeB200Error) as e:
        pkg.Pool(max_streams=8)
    assert "-3" in str(e.value)


HALF_WAVE = 148 * 14
PLAN_SIZES = (1, 13, 14, 15, 2072, 4 * HALF_WAVE, 4 * HALF_WAVE + 1, 20000, 65536, 66000, 131072, 262144, 1048576, 1048577,
              4000000)


def test_pipeline_plan_covers_every_stream_once(pkg):
    """Host logic of the host-pointer call (DESIGN 4.4): the chunk plan of a batch covers [0, n_streams) exactly once in
    order, small batches stay one chunk, large ones are tapered at both ends, and the plan never exceeds the event pool."""
    lib = pkg.load_library()
    ci = ctypes.c_int
    buf = (ci * 64)()
    assert lib.mbe_b200_pipeline_plan(0, buf, 64) == 0
    assert lib.mbe_b200_pipeline_plan(-1, buf, 64) < 0
    assert lib.mbe_b200_pipeline_plan(10, None, 64) < 0
    half_wave = HALF_WAVE
    for n in PLAN_SIZES:
        k = lib.mbe_b200_pipeline_plan(n, buf, 64)
        assert 1 <= k <= 64, (n, k)
        sizes = list(buf[:k])
        assert all(s > 0 for s in sizes) and sum(sizes) == n, (n, sizes)
        if n <= 4 * half_wave:
            assert k == 1
        assert lib.mbe_b200_pipeline_plan(n, buf, 0) == k      # count only
    # the bench workload: small pieces at both ends, half-wave multiples in between
    k = lib.mbe_b200_pipeline_plan(65536, buf, 64)
    sizes = list(buf[:k])
    assert sizes[0] == sizes[-1] == 18 * 14 and sizes[1] == sizes[-2] == 36 * 14
    assert max(sizes) == half_wave and sizes[:4] == sorted(sizes[:4]) and sizes[-4:] == sorted(sizes[-4:], reverse=True)
    assert all(s % 14 == 0 for s in sizes[:-5])


def test_pipeline_plan_under_knobs(pkg):
    """MBE_B200_CHUNKS / MBE_B200_TAPER (read once per process, so each setting runs in a child process) change how a
    host call is cut, never what it covers: every plan covers [0, n_streams) within the event pool; an out-of-range value
    is ignored; one chunk means one chunk; without a taper every chunk but the last has the same size; with one, a call
    of at least four chunks starts with pieces of TAPER x 14 x 2^i streams (below a chunk, eight at most) and ends with
    the same pieces mirrored, and the chunks between are whole."""
    import mbe_testlib as T
    chunks, tapers = (None, 1, 5, 64, 65), (None, 0, 1, 148, 149)
    knobs = lambda c, t: {k: v for k, v in (("MBE_B200_CHUNKS", c), ("MBE_B200_TAPER", t)) if v is not None}
    plans = {(c, t): T.pipeline_plans(PLAN_SIZES, knobs(c, t)) for c in chunks for t in tapers}
    for (c, t), by_n in plans.items():
        taper = 18 if t is None or t > 148 else t
        for n, sizes in by_n.items():
            where = (c, t, n, sizes)
            assert 1 <= len(sizes) <= 64 and all(s > 0 for s in sizes) and sum(sizes) == n, where
            if c == 65:
                assert sizes == plans[None, t][n], where
            if t == 149:
                assert sizes == plans[c, None][n], where
            if c == 1:
                assert len(sizes) == 1, where
            chunk = plans[c, 0][n][0]             # the taper does not change the chunk size: the untapered plan shows it
            head = [taper * 14 << i for i in range(8) if taper * 14 << i < chunk] if taper and n >= 4 * chunk else []
            assert sizes[:len(head)] == head and sizes[len(sizes) - len(head):] == head[::-1], where
            body = sizes[len(head):len(sizes) - len(head)]
            assert body and all(s == chunk for s in body[:-1]), where
            if not taper:
                assert body[-1] <= chunk, where
    assert plans[64, 0][1048576] == [16576] * 63 + [4288]
    assert plans[5, 1][1048576][:8] == [14 << i for i in range(8)]
