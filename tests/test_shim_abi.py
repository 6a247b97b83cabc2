"""Single-stream drop-in shim (SURVEY 8(f)-4), checks that need no GPU: libmbe-neo-b200shim.so loads, exports every
symbol include/mbe_b200_compat.h declares under the reference's own names, its structs have the reference's layout, and
the host-only helpers behave like the reference's (src/core/mbelib.c:61-158)."""
import ctypes
import os
import re
import subprocess
import sys

import pytest

from __graft_entry__ import ROOT

SHIM = os.path.join(ROOT, "mbelib-neo_b200", "libmbe-neo-b200shim.so")
HEADER = os.path.join(ROOT, "include", "mbe_b200_compat.h")


class SoftBit(ctypes.Structure):
    _fields_ = [("bit", ctypes.c_uint8), ("reliability", ctypes.c_uint8)]


class Result(ctypes.Structure):
    _fields_ = [("c0_errors", ctypes.c_int), ("protected_errors", ctypes.c_int), ("c4_errors", ctypes.c_int),
                ("total_errors", ctypes.c_int), ("flags", ctypes.c_uint)]


@pytest.fixture(scope="module")
def shim():
    if not os.path.exists(SHIM):
        subprocess.check_call([sys.executable, os.path.join(ROOT, "mbelib-neo_b200", "build.py")])
    return ctypes.CDLL(SHIM)


def declared():
    text = open(HEADER).read()
    names = set(re.findall(r"MBE_COMPAT_API\s+[\w\s\*]+?\b(mbe_\w+)\s*\(", text))
    names -= {"mbe_soft_bit"}
    for base in re.findall(r"^MBE_COMPAT_DATA\((mbe_\w+),", text, re.M):
        names |= {base, base + "f"}
    for base in re.findall(r"^MBE_COMPAT_FRAME\((mbe_\w+),", text, re.M):
        names |= {base + s for s in ("Frame", "Framef", "SoftFrame", "SoftFramef")}
    for codec in re.findall(r"^MBE_COMPAT_STEPS\((\w+),", text, re.M):
        names |= {"mbe_ecc%sC0" % codec, "mbe_demodulate%sData" % codec, "mbe_ecc%sData" % codec}
    return sorted(n for n in names if "##" not in n and n != "name")


def test_header_covers_the_frame_level_api():
    names = declared()
    assert len(names) == 87
    for codec in ("Imbe7200x4400", "Imbe7100x4400", "Ambe3600x2400", "Ambe3600x2450"):
        for suffix in ("Frame", "Framef", "SoftFrame", "SoftFramef"):
            assert "mbe_process%s%s" % (codec, suffix) in names
        assert "mbe_decode%sFrame" % codec in names and "mbe_decode%sSoftFrame" % codec in names


def test_shim_exports_every_declared_symbol(shim):
    for name in declared():
        assert hasattr(shim, name), "shim does not export %s" % name


def test_struct_layouts(tmp_path):
    """mbe_parms is 2604 bytes with the reference's offsets (SURVEY 8(a) Y1)."""
    src = '#include <stdio.h>\n#include <stddef.h>\n#include "mbe_b200_compat.h"\nint main(void){printf("%zu %zu %zu %zu %zu %zu %zu\\n",' \
          'sizeof(mbe_parms),offsetof(mbe_parms,Ml),offsetof(mbe_parms,gamma),offsetof(mbe_parms,previousUw),' \
          'offsetof(mbe_parms,noiseSeed),sizeof(mbe_process_result),sizeof(mbe_soft_bit));return 0;}\n'
    exe = str(tmp_path / "mbe_compat_layout")
    subprocess.run(["gcc", "-x", "c", "-", "-I" + os.path.join(ROOT, "include"), "-o", exe], input=src.encode(), check=True)
    out = subprocess.check_output([exe]).decode().split()
    assert out == ["2604", "240", "1152", "1192", "2216", "20", "2"]


def test_host_helpers(shim):
    shim.mbe_softBitFromLlr.restype = SoftBit
    shim.mbe_softBitFromLlr.argtypes = [ctypes.c_int16]
    for llr, bit, rel in ((100, 1, 100), (-100, 0, 100), (0, 0, 0), (300, 1, 255), (-32768, 0, 255)):
        s = shim.mbe_softBitFromLlr(llr)
        assert (s.bit, s.reliability) == (bit, rel)
    shim.mbe_versionString.restype = ctypes.c_char_p
    assert shim.mbe_versionString() == b"2.0.0"
    r = Result(1, 2, 0, 3, 0x10 | 0x40 | 0x80 | 0x20)
    buf = ctypes.create_string_buffer(16)
    shim.mbe_formatProcessResult(buf, ctypes.c_size_t(16), ctypes.byref(r))
    assert buf.value == b"===ETRM"
    shim.mbe_formatProcessResult(buf, ctypes.c_size_t(3), ctypes.byref(r))
    assert buf.value == b"=="
    shim.mbe_initProcessResult(ctypes.byref(r))
    assert (r.c0_errors, r.total_errors, r.flags) == (0, 0, 0)
    bits = (ctypes.c_char * 4)(0, 1, 1, 0)
    soft = (SoftBit * 4)()
    assert shim.mbe_softBitsFromHard(bits, soft, ctypes.c_size_t(4), ctypes.c_uint8(200)) == 0
    assert [(s.bit, s.reliability) for s in soft] == [(0, 200), (1, 200), (1, 200), (0, 200)]
    bad = (ctypes.c_char * 2)(0, 2)
    assert shim.mbe_softBitsFromHard(bad, soft, ctypes.c_size_t(2), ctypes.c_uint8(1)) == -2
    assert shim.mbe_softBitsFromHard(None, soft, ctypes.c_size_t(2), ctypes.c_uint8(1)) == -1
    assert shim.mbe_softBitsFromHard(bits, None, ctypes.c_size_t(2), ctypes.c_uint8(1)) == -1


def test_null_arguments_are_rejected_before_any_gpu_work(shim):
    """The reference returns MBE_STATUS_INVALID_ARGUMENT for NULL outputs/state without touching anything
    (imbe7200x4400.c:863-872,911-924); the shim does so without creating a CUDA context."""
    fn = shim.mbe_processImbe4400Data
    fn.argtypes = [ctypes.c_void_p] * 6
    assert fn(None, None, None, None, None, None) == -1
    fr = ctypes.create_string_buffer(184)
    d = ctypes.create_string_buffer(88)
    fn = shim.mbe_processImbe7200x4400Frame
    fn.argtypes = [ctypes.c_void_p] * 7
    assert fn(None, None, fr, d, None, None, None) == -1


def test_no_gpu_means_an_error_code_or_silence_never_abort():
    """SURVEY 8(b) Errors / VERDICT round 1: the reference never aborts - its int functions return
    MBE_STATUS_INVALID_ARGUMENT and its void helpers leave silence (src/core/mbelib.c:1048-1055).  Without a CUDA device (this
    test hides them) the shim must do the same: the process survives, frame calls return -1 and touch nothing, synthesis
    writes silence.  Run in a child process so that a regression (abort) fails the test instead of killing pytest."""
    code = r'''
import ctypes, sys
import numpy as np
shim = ctypes.CDLL(sys.argv[1])
vp = ctypes.c_void_p
trip = np.full((3, 2604), 7, np.uint8)
shim.mbe_initMbeParms.argtypes = [vp, vp, vp]
shim.mbe_initMbeParms(trip[0].ctypes.data, trip[1].ctypes.data, trip[2].ctypes.data)
assert (trip == 7).all(), "initMbeParms wrote something without a device"
fn = shim.mbe_processAmbe3600x2450Framef
fn.argtypes = [vp] * 7
out = np.full(160, 5.0, np.float32)
fr = np.zeros((4, 24), np.uint8)
d = np.full(49, 9, np.uint8)
rc = fn(out.ctypes.data, None, fr.ctypes.data, d.ctypes.data, trip[0].ctypes.data, trip[1].ctypes.data, trip[2].ctypes.data)
assert rc == -1, rc
assert (out == 5.0).all() and (d == 9).all() and (trip == 7).all()
shim.mbe_synthesizeSpeechf.argtypes = [vp, vp, vp]
shim.mbe_synthesizeSpeechf(out.ctypes.data, trip[0].ctypes.data, trip[1].ctypes.data)
assert (out == 0.0).all(), "synthesis without a device must leave silence"
word = np.zeros(23, np.uint8); dec = np.zeros(23, np.uint8)
shim.mbe_golay2312.argtypes = [vp, vp]
assert shim.mbe_golay2312(word.ctypes.data, dec.ctypes.data) == -1
pcm = np.full(160, 3, np.int16)
shim.mbe_floattoshort.argtypes = [vp, vp]
shim.mbe_floattoshort(out.ctypes.data, pcm.ctypes.data)
assert (pcm == 0).all()
print("survived")
'''
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", code, SHIM], env=env, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "survived" in r.stdout, (r.returncode, r.stdout[-400:], r.stderr[-800:])
    assert "no CPU fallback" in r.stderr      # it says why, once
    assert r.stderr.count("mbe_b200_create failed") == 1
