"""mbelib-neo_b200 - B200-native batched IMBE/AMBE decoder.

The product is the C-ABI shared library `libmbe_b200.so` (CUDA kernels for sm_100a + a plain-C host API,
see include/mbe_b200.h).  This package is the thin Python mirror of that ABI used by the tests and by
bench.py: it loads the library with ctypes and forwards numpy host arrays or raw device pointers.  It
contains no decoding logic and no CPU fallback - if the library or a CUDA device is missing, it raises.

Because the directory name contains a hyphen (it mirrors the reference's project name), import it through
`__graft_entry__.load_package()` (or put the repo root on sys.path and use importlib as that helper does).
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# MBE_B200_LIB lets a developer A/B an experimental build of the same library; default is the in-tree product build
LIB_PATH = os.environ.get("MBE_B200_LIB") or os.path.join(_HERE, "libmbe_b200.so")

IMBE7200X4400, IMBE7100X4400, AMBE3600X2400, AMBE3600X2450 = 0, 1, 2, 3
CODEC_BY_NAME = {"imbe7200x4400": 0, "imbe7100x4400": 1, "ambe3600x2400": 2, "ambe3600x2450": 3}
FRAME_BITS = {0: 184, 1: 168, 2: 96, 3: 96}
PARAM_BITS = {0: 88, 1: 88, 2: 49, 3: 49}
SAMPLES = 160
PARMS_BYTES = 2604

# same field order as mbe_b200_result in include/mbe_b200.h
RESULT_DTYPE = np.dtype([("status", "<i4"), ("c0_errors", "<i4"), ("protected_errors", "<i4"), ("c4_errors", "<i4"),
                         ("total_errors", "<i4"), ("flags", "<u4")])

_EXPORTS = ["mbe_b200_create", "mbe_b200_destroy", "mbe_b200_last_error", "mbe_b200_version", "mbe_b200_geometry",
            "mbe_b200_launch_count", "mbe_b200_init_streams", "mbe_b200_export_state", "mbe_b200_import_state",
            "mbe_b200_export_rng", "mbe_b200_import_rng", "mbe_b200_process_frames_dev", "mbe_b200_process_frames",
            "mbe_b200_decode_frames_dev", "mbe_b200_decode_frames", "mbe_b200_process_data_dev",
            "mbe_b200_process_data", "mbe_b200_synthesize_speech", "mbe_b200_synthesize_speech_rng", "mbe_b200_floattoshort",
            "mbe_b200_floattoshort_dev", "mbe_b200_synchronize", "mbe_b200_debug_stage_cycles",
            "mbe_b200_set_normalized_float", "mbe_b200_packed_frame_bytes", "mbe_b200_pipeline_plan", "mbe_b200_process_frames_packed_dev", "mbe_b200_process_frames_packed",
            "mbe_b200_submit_frames", "mbe_b200_wait", "mbe_b200_ecc_blocks", "mbe_b200_ecc_blocks_dev", "mbe_b200_decode_parms", "mbe_b200_spectral_amp_enhance",
            "mbe_b200_adaptive_smoothing", "mbe_b200_synthesize_tone", "mbe_b200_comfort_noise", "mbe_b200_channel_step", "mbe_b200_set_channel_map", "mbe_b200_channel_frame_bytes", "mbe_b200_pool_set_channel_map",
            "mbe_b200_device_count", "mbe_b200_pool_create", "mbe_b200_pool_destroy", "mbe_b200_pool_last_error",
            "mbe_b200_pool_shards", "mbe_b200_pool_shard", "mbe_b200_pool_init_streams", "mbe_b200_pool_export_state",
            "mbe_b200_pool_import_state", "mbe_b200_pool_process_frames", "mbe_b200_pool_process_frames_packed",
            "mbe_b200_set_kernel_path", "mbe_b200_kernel_path", "mbe_b200_set_kernel_timing", "mbe_b200_kernel_timing",
            "mbe_b200_noise_table_counters",
            "mbe_b200_host_alloc", "mbe_b200_host_free", "mbe_b200_host_register", "mbe_b200_host_unregister",
            "mbe_b200_single_frame", "mbe_b200_process_indexed_dev", "mbe_b200_process_indexed", "mbe_b200_submit_indexed",
            "mbe_b200_init_streams_indexed", "mbe_b200_export_state_indexed", "mbe_b200_import_state_indexed",
            "mbe_b200_export_rng_indexed", "mbe_b200_import_rng_indexed", "mbe_b200_pool_process_indexed",
            "mbe_b200_pool_init_streams_indexed", "mbe_b200_packed_param_bytes", "mbe_b200_process_data_indexed_dev",
            "mbe_b200_process_data_indexed", "mbe_b200_submit_data_indexed", "mbe_b200_pool_process_data_indexed"]

# `input` of the indexed calls (MBE_B200_INPUT_* of include/mbe_b200.h)
INPUT_HARD, INPUT_SOFT, INPUT_PACKED = 0, 1, 2

_lib = None


class MbeB200Error(RuntimeError):
    pass


def exported_symbols():
    return list(_EXPORTS)


def load_library():
    """dlopen libmbe_b200.so (no CUDA call is made until a context is created)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MbeB200Error("libmbe_b200.so is not built - run `python mbelib-neo_b200/build.py` "
                               "(there is no CPU fallback)")
        lib = ctypes.CDLL(LIB_PATH)
        vp, ci = ctypes.c_void_p, ctypes.c_int
        lib.mbe_b200_create.argtypes = [ctypes.POINTER(vp), ci, ci]
        lib.mbe_b200_destroy.argtypes = [vp]
        lib.mbe_b200_destroy.restype = None
        lib.mbe_b200_last_error.argtypes = [vp]
        lib.mbe_b200_last_error.restype = ctypes.c_char_p
        lib.mbe_b200_version.restype = ctypes.c_char_p
        lib.mbe_b200_launch_count.argtypes = [vp]
        lib.mbe_b200_launch_count.restype = ctypes.c_longlong
        lib.mbe_b200_geometry.argtypes = [ci, ctypes.POINTER(ci), ctypes.POINTER(ci)]
        lib.mbe_b200_init_streams.argtypes = [vp, ci, ci, vp]
        for n in ("export_state", "import_state", "export_rng", "import_rng"):
            getattr(lib, "mbe_b200_" + n).argtypes = [vp, ci, ci, vp]
        lib.mbe_b200_process_frames_dev.argtypes = [vp, ci, ci, ci, ci, ci, vp, vp, vp, vp, vp, vp]
        lib.mbe_b200_process_frames.argtypes = [vp, ci, ci, ci, ci, ci, vp, vp, vp, vp, vp]
        lib.mbe_b200_submit_frames.argtypes = [vp, ci, ci, ci, ci, ci, vp, vp, vp, vp, vp]
        lib.mbe_b200_wait.argtypes = [vp]
        lib.mbe_b200_set_normalized_float.argtypes = [vp, ci]
        lib.mbe_b200_set_kernel_path.argtypes = [vp, ci]
        lib.mbe_b200_kernel_path.argtypes = [vp]
        lib.mbe_b200_set_kernel_timing.argtypes = [vp, ci]
        lib.mbe_b200_host_alloc.argtypes = [ctypes.POINTER(vp), ctypes.c_size_t]
        lib.mbe_b200_host_free.argtypes = [vp]
        lib.mbe_b200_single_frame.argtypes = [vp, ci, ci, ci, vp, vp, vp, vp, vp, vp, vp]
        lib.mbe_b200_host_register.argtypes = [vp, ctypes.c_size_t]
        lib.mbe_b200_host_unregister.argtypes = [vp]
        lib.mbe_b200_kernel_timing.argtypes = [vp, vp, vp, vp]
        lib.mbe_b200_noise_table_counters.argtypes = [vp, vp]
        lib.mbe_b200_packed_frame_bytes.argtypes = [ci]
        lib.mbe_b200_pipeline_plan.argtypes = [ci, ctypes.POINTER(ci), ci]
        lib.mbe_b200_process_frames_packed_dev.argtypes = [vp, ci, ci, ci, ci, vp, vp, vp, vp, vp, vp]
        lib.mbe_b200_process_frames_packed.argtypes = [vp, ci, ci, ci, ci, vp, vp, vp, vp, vp]
        lib.mbe_b200_decode_frames_dev.argtypes = [vp, ci, ci, ci, vp, vp, vp, vp]
        lib.mbe_b200_decode_frames.argtypes = [vp, ci, ci, ci, vp, vp, vp]
        lib.mbe_b200_process_data_dev.argtypes = [vp, ci, ci, ci, ci, vp, vp, vp, vp, vp]
        lib.mbe_b200_process_data.argtypes = [vp, ci, ci, ci, ci, vp, vp, vp, vp]
        lib.mbe_b200_synthesize_speech.argtypes = [vp, ci, vp, vp, vp, vp, vp]
        lib.mbe_b200_synthesize_speech_rng.argtypes = [vp, ci, vp, vp, vp, vp, vp]
        lib.mbe_b200_floattoshort.argtypes = [vp, ci, vp, vp]
        lib.mbe_b200_floattoshort_dev.argtypes = [vp, ci, vp, vp, vp]
        lib.mbe_b200_synchronize.argtypes = [vp]
        lib.mbe_b200_debug_stage_cycles.argtypes = [vp, vp, ci]
        lib.mbe_b200_decode_parms.argtypes = [vp, ci, ci, vp, vp, vp, vp]
        lib.mbe_b200_spectral_amp_enhance.argtypes = [vp, ci, vp, vp]
        lib.mbe_b200_adaptive_smoothing.argtypes = [vp, ci, vp, vp]
        lib.mbe_b200_synthesize_tone.argtypes = [vp, ci, vp, vp, vp, vp]
        lib.mbe_b200_comfort_noise.argtypes = [vp, ci, vp, vp]
        lib.mbe_b200_channel_step.argtypes = [vp, ci, ci, ci, vp, vp, vp]
        lib.mbe_b200_ecc_blocks.argtypes = [vp, ci, ci, ci, vp, vp, vp]
        lib.mbe_b200_ecc_blocks_dev.argtypes = [vp, ci, ci, ci, vp, vp, vp, vp]
        lib.mbe_b200_set_channel_map.argtypes = [vp, ci, vp, ci]
        lib.mbe_b200_channel_frame_bytes.argtypes = [vp, ci]
        lib.mbe_b200_pool_set_channel_map.argtypes = [vp, ci, vp, ci]
        lib.mbe_b200_pool_create.argtypes = [ctypes.POINTER(vp), ci, vp, ci]
        lib.mbe_b200_pool_destroy.argtypes = [vp]
        lib.mbe_b200_pool_destroy.restype = None
        lib.mbe_b200_pool_last_error.argtypes = [vp]
        lib.mbe_b200_pool_last_error.restype = ctypes.c_char_p
        lib.mbe_b200_pool_shards.argtypes = [vp]
        lib.mbe_b200_pool_shard.argtypes = [vp, ci, ctypes.POINTER(ci), ctypes.POINTER(ci), ctypes.POINTER(vp)]
        lib.mbe_b200_pool_init_streams.argtypes = [vp, ci, ci, vp]
        lib.mbe_b200_pool_export_state.argtypes = [vp, ci, ci, vp]
        lib.mbe_b200_pool_import_state.argtypes = [vp, ci, ci, vp]
        lib.mbe_b200_pool_process_frames.argtypes = [vp, ci, ci, ci, ci, ci, vp, vp, vp, vp, vp]
        lib.mbe_b200_pool_process_frames_packed.argtypes = [vp, ci, ci, ci, ci, vp, vp, vp, vp, vp]
        lib.mbe_b200_process_indexed_dev.argtypes = [vp, ci, ci, vp, ci, ci, vp, vp, vp, vp, vp, vp]
        for n in ("process_indexed", "submit_indexed", "pool_process_indexed"):
            getattr(lib, "mbe_b200_" + n).argtypes = [vp, ci, ci, vp, ci, ci, vp, vp, vp, vp, vp]
        lib.mbe_b200_packed_param_bytes.argtypes = [ci]
        lib.mbe_b200_process_data_indexed_dev.argtypes = [vp, ci, ci, vp, ci, ci, vp, vp, vp, vp, vp]
        for n in ("process_data_indexed", "submit_data_indexed", "pool_process_data_indexed"):
            getattr(lib, "mbe_b200_" + n).argtypes = [vp, ci, ci, vp, ci, ci, vp, vp, vp, vp]
        for n in ("init_streams_indexed", "export_state_indexed", "import_state_indexed", "export_rng_indexed",
                  "import_rng_indexed", "pool_init_streams_indexed"):
            getattr(lib, "mbe_b200_" + n).argtypes = [vp, vp, ci, vp]
        _lib = lib
    return _lib


def packed_frame_bytes(codec):
    return (FRAME_BITS[codec] + 7) // 8


def packed_param_bytes(codec):
    """bytes of one packed parameter frame: 11 / 11 / 7 / 7"""
    return (PARAM_BITS[codec] + 7) // 8


def pack_params(codec, bits):
    """uint8 [..., param_bits] of 0/1 -> uint8 [..., packed_param_bytes(codec)], MSB first, the pad bits of the last byte
    zero (host-side data preparation for the packed parameter-bit calls)."""
    bits = np.ascontiguousarray(bits, dtype=np.uint8)
    assert bits.shape[-1] == PARAM_BITS[codec]
    return np.packbits(bits, axis=-1, bitorder="big")


def _data_indexed_args(codec, slots, bits, results, packed):
    """(slots, bits, IN/OUT results copy or None) of an indexed parameter-bit call"""
    slots = _slots(slots)
    bits = np.ascontiguousarray(bits, dtype=np.uint8)
    n, F = bits.shape[0], bits.shape[1]
    assert n == slots.size and bits.shape[2] == (packed_param_bytes(codec) if packed else PARAM_BITS[codec])
    if results is not None:
        results = np.ascontiguousarray(results, dtype=RESULT_DTYPE).reshape(n, F).copy()
    return slots, bits, results


def pack_frames(codec, frames):
    """uint8 [..., frame_bits] of 0/1 (the reference's char fr[rows][cols], row-major) -> uint8 [..., packed bytes],
    MSB first (host-side data preparation only; the decoding happens in the library)."""
    frames = np.ascontiguousarray(frames, dtype=np.uint8)
    assert frames.shape[-1] == FRAME_BITS[codec]
    return np.packbits(frames, axis=-1, bitorder="big")


def _slots(slots):
    return np.ascontiguousarray(slots, dtype=np.int32).reshape(-1)


def _indexed_outputs(codec, n, F, want_float, want_bits=True, want_results=True):
    return dict(pcm=np.zeros((n, F, SAMPLES), np.int16),
                pcmf=np.zeros((n, F, SAMPLES), np.float32) if want_float else None,
                results=np.zeros((n, F), RESULT_DTYPE) if want_results else None,
                bits=np.zeros((n, F, PARAM_BITS[codec]), np.uint8) if want_bits else None)


def _p(a):
    if a is None:
        return None
    if isinstance(a, int):
        return ctypes.c_void_p(a)
    return a.ctypes.data_as(ctypes.c_void_p)


def host_alloc(shape, dtype):
    """numpy array in page-locked host memory from mbe_b200_host_alloc (freed with host_free(array))."""
    lib = load_library()
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = ctypes.c_void_p()
    rc = lib.mbe_b200_host_alloc(ctypes.byref(p), max(n, 1))
    if rc != 0:
        raise MbeB200Error("mbe_b200_host_alloc failed (%d): %s" % (rc, lib.mbe_b200_last_error(None).decode()))
    buf = (ctypes.c_uint8 * max(n, 1)).from_address(p.value)
    a = np.frombuffer(buf, dtype=np.uint8, count=n).view(dtype).reshape(shape)
    a.flags.writeable = True
    _pinned[a.__array_interface__["data"][0]] = p.value
    return a


_pinned = {}


def host_free(a):
    lib = load_library()
    p = _pinned.pop(a.__array_interface__["data"][0], None)
    if p is not None:
        lib.mbe_b200_host_free(ctypes.c_void_p(p))


class Pool:
    """Many GPUs from one process: one context per device, the stream range sharded in contiguous blocks
    (mbe_b200_pool_*).  `devices`: list of CUDA ordinals (an ordinal may repeat), or None for every visible device."""

    def __init__(self, max_streams, devices=None):
        self.lib = load_library()
        self.h = ctypes.c_void_p()
        n = 0 if devices is None else len(devices)
        arr = (ctypes.c_int * n)(*devices) if n else None
        rc = self.lib.mbe_b200_pool_create(ctypes.byref(self.h), n, arr, int(max_streams))
        if rc != 0:
            raise MbeB200Error("mbe_b200_pool_create failed (%d): %s" % (rc, self.lib.mbe_b200_pool_last_error(None).decode()))
        self.max_streams = int(max_streams)

    def close(self):
        if self.h:
            self.lib.mbe_b200_pool_destroy(self.h)
            self.h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise MbeB200Error("%s failed (%d): %s" % (what, rc, self.lib.mbe_b200_pool_last_error(self.h).decode()))

    def shards(self):
        """[(first_stream, n_streams)] per shard."""
        out = []
        for i in range(self.lib.mbe_b200_pool_shards(self.h)):
            a, b = ctypes.c_int(), ctypes.c_int()
            self._check(self.lib.mbe_b200_pool_shard(self.h, i, ctypes.byref(a), ctypes.byref(b), None), "pool_shard")
            out.append((a.value, b.value))
        return out

    def init_streams(self, first, count, seeds=None):
        if seeds is not None:
            seeds = np.ascontiguousarray(seeds, dtype=np.uint32)
        self._check(self.lib.mbe_b200_pool_init_streams(self.h, first, count, _p(seeds)), "pool_init_streams")

    def export_state(self, first=0, count=None):
        count = self.max_streams - first if count is None else count
        out = np.zeros((count, 3, PARMS_BYTES), np.uint8)
        self._check(self.lib.mbe_b200_pool_export_state(self.h, first, count, _p(out)), "pool_export_state")
        return out

    def import_state(self, blobs, first=0):
        blobs = np.ascontiguousarray(blobs, dtype=np.uint8).reshape(-1, 3, PARMS_BYTES)
        self._check(self.lib.mbe_b200_pool_import_state(self.h, first, blobs.shape[0], _p(blobs)), "pool_import_state")

    def set_channel_map(self, codec, channel_map=None):
        """mbe_b200_pool_set_channel_map: the same interleave schedule on every shard (None: identity)."""
        if channel_map is None:
            self._check(self.lib.mbe_b200_pool_set_channel_map(self.h, codec, None, 0), "pool_set_channel_map")
        else:
            m = np.ascontiguousarray(channel_map, dtype=np.uint16)
            self._check(self.lib.mbe_b200_pool_set_channel_map(self.h, codec, _p(m), int(m.size)), "pool_set_channel_map")

    def process_frames(self, codec, frames, soft=False, first_stream=0, want_float=False, packed=False):
        frames = np.ascontiguousarray(frames, dtype=np.uint8)
        S, F = frames.shape[0], frames.shape[1]
        pcm = np.zeros((S, F, SAMPLES), np.int16)
        pcmf = np.zeros((S, F, SAMPLES), np.float32) if want_float else None
        res = np.zeros((S, F), RESULT_DTYPE)
        bits = np.zeros((S, F, PARAM_BITS[codec]), np.uint8)
        if packed:
            rc = self.lib.mbe_b200_pool_process_frames_packed(self.h, codec, first_stream, S, F, _p(frames), _p(pcm), _p(pcmf),
                                                              _p(res), _p(bits))
        else:
            rc = self.lib.mbe_b200_pool_process_frames(self.h, codec, int(bool(soft)), first_stream, S, F, _p(frames), _p(pcm),
                                                       _p(pcmf), _p(res), _p(bits))
        self._check(rc, "pool_process_frames")
        return dict(pcm=pcm, pcmf=pcmf, results=res, bits=bits)

    def init_streams_indexed(self, slots, seeds=None):
        """mbe_b200_pool_init_streams_indexed: init_streams of the listed global slots (seeds[i] for slots[i])."""
        slots = _slots(slots)
        if seeds is not None:
            seeds = np.ascontiguousarray(seeds, dtype=np.uint32)
            assert seeds.size == slots.size
        self._check(self.lib.mbe_b200_pool_init_streams_indexed(self.h, _p(slots), slots.size, _p(seeds)),
                    "pool_init_streams_indexed")

    def process_indexed(self, codec, slots, frames, input=INPUT_HARD, want_float=False):
        """mbe_b200_pool_process_indexed: element i of `frames` ([n][F][...]) is global slot slots[i]."""
        slots = _slots(slots)
        frames = np.ascontiguousarray(frames, dtype=np.uint8)
        n, F = frames.shape[0], frames.shape[1]
        assert n == slots.size
        out = _indexed_outputs(codec, n, F, want_float)
        self._check(self.lib.mbe_b200_pool_process_indexed(self.h, codec, int(input), _p(slots), n, F, _p(frames),
                                                           _p(out["pcm"]), _p(out["pcmf"]), _p(out["results"]),
                                                           _p(out["bits"])), "pool_process_indexed")
        return out

    def process_data_indexed(self, codec, slots, bits, results=None, packed=False, want_float=False):
        """mbe_b200_pool_process_data_indexed: element i of `bits` ([n][F][88|49], or [n][F][11|7] packed) and of
        `results` (IN/OUT decode context, None = none) is global slot slots[i].  Returns the dict process_data returns."""
        slots, bits, results = _data_indexed_args(codec, slots, bits, results, packed)
        n, F = bits.shape[0], bits.shape[1]
        pcm = np.zeros((n, F, SAMPLES), np.int16)
        pcmf = np.zeros((n, F, SAMPLES), np.float32) if want_float else None
        self._check(self.lib.mbe_b200_pool_process_data_indexed(self.h, codec, int(bool(packed)), _p(slots), n, F, _p(bits),
                                                                _p(results), _p(pcm), _p(pcmf)), "pool_process_data_indexed")
        return dict(pcm=pcm, pcmf=pcmf, results=results)


class Decoder:
    """One context = one GPU + a pool of `max_streams` device-resident voice-stream states."""

    def __init__(self, max_streams, device=0):
        self.lib = load_library()
        self.h = ctypes.c_void_p()
        rc = self.lib.mbe_b200_create(ctypes.byref(self.h), int(device), int(max_streams))
        if rc != 0:
            raise MbeB200Error("mbe_b200_create failed (%d): %s" % (rc, self.lib.mbe_b200_last_error(None).decode()))
        self.max_streams = int(max_streams)
        self.device = int(device)

    def close(self):
        if self.h:
            self.lib.mbe_b200_destroy(self.h)
            self.h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise MbeB200Error("%s failed (%d): %s" % (what, rc, self.lib.mbe_b200_last_error(self.h).decode()))

    @property
    def launches(self):
        return int(self.lib.mbe_b200_launch_count(self.h))

    # ---- state ----
    def init_streams(self, first=0, count=None, seeds=None):
        count = self.max_streams - first if count is None else count
        if seeds is not None:
            seeds = np.ascontiguousarray(seeds, dtype=np.uint32)
            assert seeds.size == count
        self._check(self.lib.mbe_b200_init_streams(self.h, first, count, _p(seeds)), "init_streams")

    def export_state(self, first=0, count=None):
        count = self.max_streams - first if count is None else count
        out = np.zeros((count, 3, PARMS_BYTES), np.uint8)
        self._check(self.lib.mbe_b200_export_state(self.h, first, count, _p(out)), "export_state")
        return out

    def import_state(self, blobs, first=0):
        blobs = np.ascontiguousarray(blobs, dtype=np.uint8).reshape(-1, 3, PARMS_BYTES)
        self._check(self.lib.mbe_b200_import_state(self.h, first, blobs.shape[0], _p(blobs)), "import_state")

    def export_rng(self, first=0, count=None):
        count = self.max_streams - first if count is None else count
        out = np.zeros((count, 4), np.uint32)
        self._check(self.lib.mbe_b200_export_rng(self.h, first, count, _p(out)), "export_rng")
        return out

    def import_rng(self, words, first=0):
        words = np.ascontiguousarray(words, dtype=np.uint32).reshape(-1, 4)
        self._check(self.lib.mbe_b200_import_rng(self.h, first, words.shape[0], _p(words)), "import_rng")

    # ---- indexed state calls: host slot lists, element i <-> slots[i] ----
    def init_streams_indexed(self, slots, seeds=None):
        slots = _slots(slots)
        if seeds is not None:
            seeds = np.ascontiguousarray(seeds, dtype=np.uint32)
            assert seeds.size == slots.size
        self._check(self.lib.mbe_b200_init_streams_indexed(self.h, _p(slots), slots.size, _p(seeds)), "init_streams_indexed")

    def export_state_indexed(self, slots):
        slots = _slots(slots)
        out = np.zeros((slots.size, 3, PARMS_BYTES), np.uint8)
        self._check(self.lib.mbe_b200_export_state_indexed(self.h, _p(slots), slots.size, _p(out)), "export_state_indexed")
        return out

    def import_state_indexed(self, slots, blobs):
        slots = _slots(slots)
        blobs = np.ascontiguousarray(blobs, dtype=np.uint8).reshape(-1, 3, PARMS_BYTES)
        assert blobs.shape[0] == slots.size
        self._check(self.lib.mbe_b200_import_state_indexed(self.h, _p(slots), slots.size, _p(blobs)), "import_state_indexed")

    def export_rng_indexed(self, slots):
        slots = _slots(slots)
        out = np.zeros((slots.size, 4), np.uint32)
        self._check(self.lib.mbe_b200_export_rng_indexed(self.h, _p(slots), slots.size, _p(out)), "export_rng_indexed")
        return out

    def import_rng_indexed(self, slots, words):
        slots = _slots(slots)
        words = np.ascontiguousarray(words, dtype=np.uint32).reshape(-1, 4)
        assert words.shape[0] == slots.size
        self._check(self.lib.mbe_b200_import_rng_indexed(self.h, _p(slots), slots.size, _p(words)), "import_rng_indexed")

    # ---- indexed batches: element i of frames / outputs is stream slot slots[i] ----
    def process_indexed(self, codec, slots, frames, input=INPUT_HARD, want_float=False, want_bits=True, want_results=True):
        """frames: uint8 [n][F][bits] (INPUT_HARD), [n][F][bits][2] (INPUT_SOFT) or [n][F][channel bytes] (INPUT_PACKED)."""
        slots = _slots(slots)
        frames = np.ascontiguousarray(frames, dtype=np.uint8)
        n, F = frames.shape[0], frames.shape[1]
        assert n == slots.size
        out = _indexed_outputs(codec, n, F, want_float, want_bits, want_results)
        self._check(self.lib.mbe_b200_process_indexed(self.h, codec, int(input), _p(slots), n, F, _p(frames), _p(out["pcm"]),
                                                      _p(out["pcmf"]), _p(out["results"]), _p(out["bits"])),
                    "process_indexed")
        return out

    def submit_indexed(self, codec, slots, frames, out, input=INPUT_HARD):
        """Asynchronous process_indexed: `slots`, `frames` and the arrays of `out` (dict with pcm / pcmf / results / bits,
        any may be missing) must stay alive and untouched until wait()."""
        assert slots.dtype == np.int32 and slots.flags["C_CONTIGUOUS"]
        n, F = frames.shape[0], frames.shape[1]
        self._check(self.lib.mbe_b200_submit_indexed(self.h, codec, int(input), _p(slots), n, F, _p(frames),
                                                     _p(out.get("pcm")), _p(out.get("pcmf")), _p(out.get("results")),
                                                     _p(out.get("bits"))), "submit_indexed")

    def process_indexed_dev(self, codec, input, d_slots, n, n_frames, d_in, d_pcm, d_pcmf=0, d_results=0, d_bits=0,
                            cuda_stream=0):
        """All pointers are raw device addresses (ints), d_slots int32 [n]; asynchronous on `cuda_stream`."""
        self._check(self.lib.mbe_b200_process_indexed_dev(self.h, codec, int(input), _p(d_slots), n, n_frames, _p(d_in),
                                                          _p(d_pcm or None), _p(d_pcmf or None), _p(d_results or None),
                                                          _p(d_bits or None), _p(cuda_stream or None)),
                    "process_indexed_dev")

    # ---- indexed parameter-bit batches (mbe_process<Codec>Data): element i of bits / results / outputs is slot slots[i] ----
    def process_data_indexed(self, codec, slots, bits, results=None, packed=False, want_float=False):
        """bits: uint8 [n][F][88|49] one byte per bit, or [n][F][packed_param_bytes(codec)] with packed=True (see
        pack_params); results: the IN/OUT decode context [n][F] (None = none).  Returns the dict process_data returns."""
        slots, bits, results = _data_indexed_args(codec, slots, bits, results, packed)
        n, F = bits.shape[0], bits.shape[1]
        pcm = np.zeros((n, F, SAMPLES), np.int16)
        pcmf = np.zeros((n, F, SAMPLES), np.float32) if want_float else None
        self._check(self.lib.mbe_b200_process_data_indexed(self.h, codec, int(bool(packed)), _p(slots), n, F, _p(bits),
                                                           _p(results), _p(pcm), _p(pcmf)), "process_data_indexed")
        return dict(pcm=pcm, pcmf=pcmf, results=results)

    def submit_data_indexed(self, codec, slots, bits, out, packed=False):
        """Asynchronous process_data_indexed: `slots`, `bits` and the arrays of `out` (dict with pcm / pcmf / results, any
        may be missing; results holds the decode context in and the results out) must stay alive and untouched until
        wait()."""
        assert slots.dtype == np.int32 and slots.flags["C_CONTIGUOUS"]
        n, F = bits.shape[0], bits.shape[1]
        self._check(self.lib.mbe_b200_submit_data_indexed(self.h, codec, int(bool(packed)), _p(slots), n, F, _p(bits),
                                                          _p(out.get("results")), _p(out.get("pcm")), _p(out.get("pcmf"))),
                    "submit_data_indexed")

    def process_data_indexed_dev(self, codec, packed, d_slots, n, n_frames, d_bits, d_results_inout, d_pcm, d_pcmf=0,
                                 cuda_stream=0):
        """All pointers are raw device addresses (ints, 0 = NULL), d_slots int32 [n]; asynchronous on `cuda_stream`."""
        self._check(self.lib.mbe_b200_process_data_indexed_dev(self.h, codec, int(bool(packed)), _p(d_slots), n, n_frames,
                                                               _p(d_bits), _p(d_results_inout or None), _p(d_pcm or None),
                                                               _p(d_pcmf or None), _p(cuda_stream or None)),
                    "process_data_indexed_dev")

    # ---- hot path, host buffers ----
    def process_frames(self, codec, frames, soft=False, first_stream=0, want_float=False, want_bits=True,
                       want_results=True, out_pcm=None):
        """frames: uint8 [S][F][bits] (hard) or [S][F][bits][2] (soft). Returns dict of numpy arrays."""
        frames = np.ascontiguousarray(frames, dtype=np.uint8)
        S, F = frames.shape[0], frames.shape[1]
        pcm = out_pcm if out_pcm is not None else np.zeros((S, F, SAMPLES), np.int16)
        pcmf = np.zeros((S, F, SAMPLES), np.float32) if want_float else None
        res = np.zeros((S, F), RESULT_DTYPE) if want_results else None
        bits = np.zeros((S, F, PARAM_BITS[codec]), np.uint8) if want_bits else None
        self._check(self.lib.mbe_b200_process_frames(self.h, codec, int(bool(soft)), first_stream, S, F, _p(frames),
                                                     _p(pcm), _p(pcmf), _p(res), _p(bits)), "process_frames")
        return dict(pcm=pcm, pcmf=pcmf, results=res, bits=bits)

    def set_channel_map(self, codec, channel_map=None):
        """channel_map[k] = frame position (r*cols + c) of transmitted bit k of the bit-packed input; None = identity."""
        if channel_map is None:
            self._check(self.lib.mbe_b200_set_channel_map(self.h, codec, None, 0), "set_channel_map")
        else:
            m = np.ascontiguousarray(channel_map, dtype=np.uint16)
            self._check(self.lib.mbe_b200_set_channel_map(self.h, codec, _p(m), int(m.size)), "set_channel_map")

    def channel_frame_bytes(self, codec):
        return int(self.lib.mbe_b200_channel_frame_bytes(self.h, codec))

    def submit_frames(self, codec, frames, out, soft=False, first_stream=0):
        """Asynchronous process_frames: `frames` and the arrays of `out` (dict with pcm / results / bits, any may be missing)
        must stay alive and untouched until wait()."""
        S, F = frames.shape[0], frames.shape[1]
        self._check(self.lib.mbe_b200_submit_frames(self.h, codec, int(bool(soft)), first_stream, S, F, _p(frames),
                                                    _p(out.get("pcm")), _p(out.get("pcmf")), _p(out.get("results")),
                                                    _p(out.get("bits"))), "submit_frames")

    def wait(self):
        self._check(self.lib.mbe_b200_wait(self.h), "wait")

    def set_kernel_path(self, path):
        """0: one fused kernel per batch; 1: parameter kernel + synthesis kernel (bit-identical results)."""
        self._check(self.lib.mbe_b200_set_kernel_path(self.h, int(path)), "set_kernel_path")

    def kernel_path(self):
        return int(self.lib.mbe_b200_kernel_path(self.h))

    def set_kernel_timing(self, enable):
        self._check(self.lib.mbe_b200_set_kernel_timing(self.h, int(bool(enable))), "set_kernel_timing")

    def kernel_timing(self):
        """{kind: (ms, launches)} for kinds parameter / bank / unvoiced, and the bank kernel's work counters."""
        ms = np.zeros(3, np.float64)
        n = np.zeros(3, np.int64)
        cnt = np.zeros(4, np.uint64)
        self._check(self.lib.mbe_b200_kernel_timing(self.h, _p(ms), _p(n), _p(cnt)), "kernel_timing")
        names = ("parameter", "bank", "unvoiced")
        return ({names[i]: (float(ms[i]), int(n[i])) for i in range(3)},
                dict(slots=int(cnt[0]), interpolated=int(cnt[1]), frames=int(cnt[2])))

    def noise_table_counters(self):
        """Unvoiced-kernel frames since set_kernel_timing(True): (noise spectra read from the table, computed in the kernel)."""
        cnt = np.zeros(2, np.uint64)
        self._check(self.lib.mbe_b200_noise_table_counters(self.h, _p(cnt)), "noise_table_counters")
        return int(cnt[0]), int(cnt[1])

    def set_normalized_float(self, enable):
        self._check(self.lib.mbe_b200_set_normalized_float(self.h, int(bool(enable))), "set_normalized_float")

    def process_frames_packed(self, codec, packed, first_stream=0, want_float=False, want_bits=True, want_results=True):
        """packed: uint8 [S][F][packed_frame_bytes(codec)] hard bits, eight per byte, MSB first (see pack_frames)."""
        packed = np.ascontiguousarray(packed, dtype=np.uint8)
        S, F = packed.shape[0], packed.shape[1]
        pcm = np.zeros((S, F, SAMPLES), np.int16)
        pcmf = np.zeros((S, F, SAMPLES), np.float32) if want_float else None
        res = np.zeros((S, F), RESULT_DTYPE) if want_results else None
        bits = np.zeros((S, F, PARAM_BITS[codec]), np.uint8) if want_bits else None
        self._check(self.lib.mbe_b200_process_frames_packed(self.h, codec, first_stream, S, F, _p(packed), _p(pcm),
                                                            _p(pcmf), _p(res), _p(bits)), "process_frames_packed")
        return dict(pcm=pcm, pcmf=pcmf, results=res, bits=bits)

    def process_frames_packed_dev(self, codec, first_stream, n_streams, n_frames, d_packed, d_pcm, d_pcmf=0,
                                  d_results=0, d_bits=0, cuda_stream=0):
        self._check(self.lib.mbe_b200_process_frames_packed_dev(self.h, codec, first_stream, n_streams, n_frames,
                                                                _p(d_packed), _p(d_pcm or None), _p(d_pcmf or None),
                                                                _p(d_results or None), _p(d_bits or None),
                                                                _p(cuda_stream or None)), "process_frames_packed_dev")

    def process_frames_dev(self, codec, soft, first_stream, n_streams, n_frames, d_frames, d_pcm, d_pcmf=0,
                           d_results=0, d_bits=0, cuda_stream=0):
        """All pointers are raw device addresses (ints); asynchronous on `cuda_stream`."""
        self._check(self.lib.mbe_b200_process_frames_dev(self.h, codec, int(bool(soft)), first_stream, n_streams,
                                                         n_frames, _p(d_frames), _p(d_pcm or None), _p(d_pcmf or None),
                                                         _p(d_results or None), _p(d_bits or None),
                                                         _p(cuda_stream or None)), "process_frames_dev")

    def decode_frames(self, codec, frames, soft=False):
        frames = np.ascontiguousarray(frames, dtype=np.uint8)
        n = frames.size // (FRAME_BITS[codec] * (2 if soft else 1))
        bits = np.zeros((n, PARAM_BITS[codec]), np.uint8)
        res = np.zeros(n, RESULT_DTYPE)
        self._check(self.lib.mbe_b200_decode_frames(self.h, codec, int(bool(soft)), n, _p(frames), _p(bits), _p(res)),
                    "decode_frames")
        return bits, res

    def decode_parms(self, codec, bits, cur, prev):
        """bits uint8 [n][88|49]; cur/prev uint8 [n][2604] blobs, updated in place.  Returns status int32 [n]."""
        bits = np.ascontiguousarray(bits, dtype=np.uint8)
        n = bits.shape[0]
        status = np.zeros(n, np.int32)
        self._check(self.lib.mbe_b200_decode_parms(self.h, codec, n, _p(bits), _p(cur), _p(prev), _p(status)), "decode_parms")
        return status

    def spectral_amp_enhance(self, cur):
        rm0 = np.zeros(cur.shape[0], np.float32)
        self._check(self.lib.mbe_b200_spectral_amp_enhance(self.h, cur.shape[0], _p(cur), _p(rm0)), "spectral_amp_enhance")
        return rm0

    def adaptive_smoothing(self, cur, prev):
        self._check(self.lib.mbe_b200_adaptive_smoothing(self.h, cur.shape[0], _p(cur), _p(prev)), "adaptive_smoothing")

    def synthesize_tone(self, cur, bits49=None, dstar_id=None):
        n = cur.shape[0]
        pcmf = np.zeros((n, SAMPLES), np.float32)
        if bits49 is not None:
            bits49 = np.ascontiguousarray(bits49, dtype=np.uint8)
        if dstar_id is not None:
            dstar_id = np.ascontiguousarray(dstar_id, dtype=np.int32)
        self._check(self.lib.mbe_b200_synthesize_tone(self.h, n, _p(bits49), _p(dstar_id), _p(cur), _p(pcmf)), "synthesize_tone")
        return pcmf

    def comfort_noise(self, rng_words):
        """rng_words uint32 [n][4] (as export_rng), updated in place."""
        n = rng_words.shape[0]
        pcmf = np.zeros((n, SAMPLES), np.float32)
        self._check(self.lib.mbe_b200_comfort_noise(self.h, n, _p(rng_words), _p(pcmf)), "comfort_noise")
        return pcmf

    def channel_step(self, codec, step, frames=None, bits=None):
        """step 0/1: frames uint8 [n][frame_bits] updated in place; 2: frames -> bits; 3: bits [n][88] in place."""
        n = (frames if frames is not None else bits).shape[0]
        status = np.zeros(n, np.int32)
        self._check(self.lib.mbe_b200_channel_step(self.h, codec, step, n, _p(frames), _p(bits), _p(status)), "channel_step")
        return status

    def ecc_blocks(self, code, words, soft=False):
        """words: uint8 [n][len] bits (or [n][len][2] soft bits), len = 23 (code 0) or 15.  Returns (out [n][len], status [n])."""
        words = np.ascontiguousarray(words, dtype=np.uint8)
        n = words.shape[0]
        ln = 23 if code == 0 else 15
        out = np.zeros((n, ln), np.uint8)
        status = np.zeros(n, np.int32)
        self._check(self.lib.mbe_b200_ecc_blocks(self.h, code, int(bool(soft)), n, _p(words), _p(out), _p(status)), "ecc_blocks")
        return out, status

    def process_data(self, codec, bits, results=None, first_stream=0, want_float=False):
        bits = np.ascontiguousarray(bits, dtype=np.uint8)
        S, F = bits.shape[0], bits.shape[1]
        pcm = np.zeros((S, F, SAMPLES), np.int16)
        pcmf = np.zeros((S, F, SAMPLES), np.float32) if want_float else None
        if results is not None:
            results = np.ascontiguousarray(results, dtype=RESULT_DTYPE).reshape(S, F).copy()
        self._check(self.lib.mbe_b200_process_data(self.h, codec, first_stream, S, F, _p(bits), _p(results), _p(pcm),
                                                   _p(pcmf)), "process_data")
        return dict(pcm=pcm, pcmf=pcmf, results=results)

    def synthesize_speech(self, cur, prev, seeds=None):
        """cur/prev: uint8 [n][2604] mbe_parms blobs, updated in place. Returns (pcmf, pcm)."""
        n = cur.shape[0]
        assert cur.flags["C_CONTIGUOUS"] and prev.flags["C_CONTIGUOUS"] and cur.dtype == np.uint8
        pcmf = np.zeros((n, SAMPLES), np.float32)
        pcm = np.zeros((n, SAMPLES), np.int16)
        if seeds is not None:
            seeds = np.ascontiguousarray(seeds, dtype=np.uint32)
        self._check(self.lib.mbe_b200_synthesize_speech(self.h, n, _p(cur), _p(prev), _p(seeds), _p(pcmf), _p(pcm)),
                    "synthesize_speech")
        return pcmf, pcm

    def floattoshort(self, x):
        x = np.ascontiguousarray(x, dtype=np.float32).reshape(-1, SAMPLES)
        out = np.zeros(x.shape, np.int16)
        self._check(self.lib.mbe_b200_floattoshort(self.h, x.shape[0], _p(x), _p(out)), "floattoshort")
        return out

    def debug_stage_cycles(self, reset=True):
        out = np.zeros(16, np.uint64)
        self._check(self.lib.mbe_b200_debug_stage_cycles(self.h, _p(out), int(reset)), "debug_stage_cycles")
        return out

    def synchronize(self):
        self._check(self.lib.mbe_b200_synchronize(self.h), "synchronize")
