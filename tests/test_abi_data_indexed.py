"""C-ABI checks of the indexed parameter-bit calls that need no GPU: the symbols are declared and exported, the packed
frame size per codec, the packing convention of the Python helper, and the argument checks that come before any device
work."""
import ctypes
import os
import re

import numpy as np
import pytest

from __graft_entry__ import ROOT, load_package

NEW = ("mbe_b200_packed_param_bytes", "mbe_b200_process_data_indexed_dev", "mbe_b200_process_data_indexed",
       "mbe_b200_submit_data_indexed", "mbe_b200_pool_process_data_indexed")


@pytest.fixture(scope="module")
def pkg():
    p = load_package()
    if not os.path.exists(p.LIB_PATH):
        import subprocess
        import sys
        subprocess.check_call([sys.executable, os.path.join(ROOT, "mbelib-neo_b200", "build.py")])
    return p


def test_declared_and_exported(pkg):
    text = open(os.path.join(ROOT, "include", "mbe_b200.h")).read()
    declared = set(re.findall(r"MBE_B200_API\s+[\w\s\*]+?\b(mbe_b200_\w+)\s*\(", text))
    lib = pkg.load_library()
    for name in NEW:
        assert name in declared, name
        assert hasattr(lib, name), name
        assert name in pkg.exported_symbols(), name


def test_packed_param_bytes(pkg):
    lib = pkg.load_library()
    for codec, want in {0: 11, 1: 11, 2: 7, 3: 7}.items():
        assert lib.mbe_b200_packed_param_bytes(codec) == want
        assert pkg.packed_param_bytes(codec) == want
    for bad in (-1, 4, 99):
        assert lib.mbe_b200_packed_param_bytes(bad) == -1


def test_pack_params_is_msb_first(pkg):
    rng = np.random.default_rng(7)
    for codec in range(4):
        pb = pkg.PARAM_BITS[codec]
        bits = rng.integers(0, 2, size=(3, 2, pb), dtype=np.uint8)
        packed = pkg.pack_params(codec, bits)
        assert packed.shape == (3, 2, pkg.packed_param_bytes(codec))
        k = np.arange(pb)
        assert np.array_equal((packed[..., k >> 3] >> (7 - (k & 7))) & 1, bits)


def test_argument_checks_without_a_device(pkg):
    """Calls without a context or pool fail with MBE_B200_E_ARG before any device work."""
    lib = pkg.load_library()
    slots = (ctypes.c_int32 * 2)(0, 1)
    bits = (ctypes.c_uint8 * 256)()
    pcm = (ctypes.c_int16 * (2 * 160))()
    for packed in (0, 1, 2, -1):
        assert lib.mbe_b200_process_data_indexed(None, 0, packed, slots, 2, 1, bits, None, pcm, None) == -1
        assert lib.mbe_b200_submit_data_indexed(None, 0, packed, slots, 2, 1, bits, None, pcm, None) == -1
        assert lib.mbe_b200_process_data_indexed_dev(None, 0, packed, slots, 2, 1, bits, None, pcm, None, None) == -1
        assert lib.mbe_b200_pool_process_data_indexed(None, 0, packed, slots, 2, 1, bits, None, pcm, None) == -1
    # empty calls need a context too
    assert lib.mbe_b200_process_data_indexed(None, 0, 0, None, 0, 0, bits, None, None, None) == -1
