"""The host code that decides where each kernel runs, under every tuning knob, against the CPU oracle.

A host-pointer frame call cuts its batch into pipeline chunks spread over compute streams; on the multi-kernel path every
launch is further cut into descriptor ranges (as many streams as have their descriptors in MBE_B200_DESC_MB MiB), and a
device-resident call on a stream that is not a pipeline stream forks its ranges over MBE_B200_AUX internal streams.  Each
piece offsets the frame / PCM / result pointers (io_base), the state slots and, for indexed calls, the slot list and claim
tags (slot_base).  With the default knobs a batch needs more than 8 288 streams to be cut into chunks and about 85 000 to be
cut into ranges.  The knobs are read once per process, so each setting runs the library in a child process
(tests/helpers/knob_child.py); a 1 MiB descriptor budget brings the range cuts down to 42 - 113 streams, small enough for the
oracle.  Every output is compared with the oracle bit for bit - int16 PCM, float PCM, results, parameter bits, final
mbe_parms triplets and RNG words - and every call's launch count shows that the setting took effect."""
import json
import os

import numpy as np
import pytest

import mbe_testlib as T

pytestmark = pytest.mark.gpu

M, FIRST, S = 12000, 37, 9000          # pool size, first stream of the contiguous calls, streams per call
CUTS3, CUTS0 = [(0, 3), (3, 8)], [(0, 2), (2, 6)]   # every row decodes its frames in two calls of different lengths
S_SOFT = 600
DESC_WORDS = 768                       # uint32 words of descriptor per stream-frame on the multi-kernel path (mbe_split.cuh)
MAX_CHUNKS = 64                        # pipeline chunks of one host call at most (mbe_b200_pipeline_plan)

SETTINGS = [
    ("default", {}),
    ("desc1", {"MBE_B200_DESC_MB": 1}),
    # every range on one internal stream: one descriptor buffer reused back to back
    ("desc1-aux1", {"MBE_B200_DESC_MB": 1, "MBE_B200_AUX": 1}),
    # a range count that is not a multiple of the internal streams; every pipeline chunk on one compute stream
    ("desc1-aux3-kstreams1", {"MBE_B200_DESC_MB": 1, "MBE_B200_AUX": 3, "MBE_B200_KSTREAMS": 1}),
    # an explicit chunk count: chunks are not rounded to whole ranges, so the last range of every chunk is ragged
    ("desc1-chunks3", {"MBE_B200_DESC_MB": 1, "MBE_B200_CHUNKS": 3}),
    ("chunks64-taper0-kstreams3", {"MBE_B200_CHUNKS": 64, "MBE_B200_TAPER": 0, "MBE_B200_KSTREAMS": 3}),
    # eight taper pieces at each end, the smallest 14 streams
    ("chunks5-taper1", {"MBE_B200_CHUNKS": 5, "MBE_B200_TAPER": 1}),
    # the fused kernel as the context default
    ("fused-chunks64-taper1", {"MBE_B200_SPLIT": 0, "MBE_B200_CHUNKS": 64, "MBE_B200_TAPER": 1}),
]


@pytest.fixture(scope="module")
def case(tmp_path_factory):
    """The seeded inputs (written once for every child) and the oracle's answers."""
    rng = np.random.default_rng(0x6B0B)
    frames3 = T.mixed_frames(3, S, 8, 0x6B03)
    frames0 = T.mixed_frames(0, S, 6, 0x6B00)
    soft0 = T.soften(T.mixed_frames(0, S_SOFT, 6, 0x6B01), rng, flip_p=0.05)
    seeds = T.stream_seeds(M, 0x6B5)
    # indexed calls: a permutation of 9 000 of the 12 000 slots; element 8 900 (the last pipeline chunk) repeats element
    # 100's slot (the first chunk), elements 4 000 and 6 000 name slots -1 and M: those three are rejected
    slots = rng.permutation(M)[:S].astype(np.int32)
    slots[8900], slots[4000], slots[6000] = slots[100], -1, M
    accepted = np.ones(S, bool)
    accepted[[8900, 4000, 6000]] = False
    idle = np.setdiff1d(np.arange(M), slots[accepted]).astype(np.int32)
    inp = str(tmp_path_factory.mktemp("knobs") / "in.npz")
    np.savez(inp, max_streams=M, first_stream=FIRST, seeds=seeds, frames3=frames3, frames0=frames0, soft0=soft0,
             cuts3=np.array(CUTS3), cuts0=np.array(CUTS0), slots=slots, accepted=accepted, idle_slots=idle)
    o = T.load_oracle().mbo_run
    want = {}
    for key, codec, soft, fr in (("w3", 3, 0, frames3), ("w0", 0, 0, frames0), ("ws", 0, 1, soft0)):
        sd = seeds[FIRST:FIRST + fr.shape[0]]
        want[key] = T.run_cpu(o, codec, soft, fr, sd, n_threads=16)
        want[key]["rng"] = T.oracle_rng_words(codec, soft, fr, sd, n_threads=16)
    return dict(inp=inp, want=want, accepted=accepted, default_plans=T.pipeline_plans([S, S_SOFT], {}))


def _diff(failures, tag, got, want):
    got, want = np.asarray(got), np.asarray(want)
    if got.dtype == np.float32:
        got, want = got.view(np.uint32), want.view(np.uint32)
    if got.shape != want.shape:
        failures.append("%s: shape %s, oracle %s" % (tag, got.shape, want.shape))
        return
    ne = got != want
    if ne.any():
        failures.append("%s: %d of %d values differ, the first at %s" % (tag, int(ne.sum()), ne.size,
                                                                          tuple(int(i) for i in np.argwhere(ne)[0])))


def _expected_launches(call, meta, knobs):
    """(least, most) launches of one call under `knobs`."""
    extra = int(call["indexed"])                    # the claim launch over the whole slot list
    plan = meta["plans"][str(call["n"])]
    if meta["kernel_path"] == 0:                    # fused: one launch per pipeline chunk or per device-resident call
        k = (len(plan) if call["pipelined"] else 1) + extra
        return k, k
    # multi-kernel path: parameter, bank and unvoiced kernel per descriptor range.  A range holds as many streams as have
    # their descriptors (n_frames x DESC_WORDS x 4 bytes each) in the budget (split_cap_streams).  1 MiB holds 42 - 113
    # streams of 8 - 3 frames: below one wave of the parameter kernel, so not rounded down to whole waves, and above its
    # floor of one block (14 streams).  The default 2 GiB holds 87 381 streams of 8 frames, at most a wave (5 328) less
    # after that rounding: every call here is one range per launch.
    if "MBE_B200_DESC_MB" in knobs:
        cap = (int(knobs["MBE_B200_DESC_MB"]) << 20) // (call["frames"] * DESC_WORDS * 4)
        assert 14 <= cap < 148 * 18 * 2
    else:
        cap = 1 << 30
    ranges = lambda ns: -(-ns // cap)
    if not call["pipelined"]:                       # one launch over the whole call
        k = 3 * ranges(call["n"]) + extra
        return k, k
    if cap > call["n"] or "MBE_B200_CHUNKS" in knobs:
        k = 3 * sum(ranges(ns) for ns in plan) + extra       # the chunks are the plan's
        return k, k
    # Multi-kernel path, no explicit chunk count: frames_host_impl rounds every chunk that holds a whole range to whole
    # ranges, which the context-free plan does not show.  Each range still holds at most `cap` streams, and each chunk adds
    # at most one partial range.  (9 000 x 3 frames under 1 MiB: 83 ranges in chunks of 2 034 streams, tapered.)
    return 3 * ranges(call["n"]) + extra, 3 * (ranges(call["n"]) + MAX_CHUNKS - 1) + extra


@pytest.mark.parametrize("name,knobs", SETTINGS, ids=[s[0] for s in SETTINGS])
def test_host_paths_under_knobs_equal_the_oracle(case, tmp_path, name, knobs):
    out = str(tmp_path / "out.npz")
    log = T.run_knob_child(["run", case["inp"], out], knobs, timeout=900)
    z = np.load(out)
    meta = json.loads(str(z["meta"]))
    failures = []

    # the settings reached the library
    assert {k: v for k, v in meta["env"].items() if k in T.KNOBS} == {k: str(v) for k, v in knobs.items()}
    assert meta["kernel_path"] == (0 if knobs.get("MBE_B200_SPLIT") == 0 else 1)
    if meta["sm_count"] == 148:                    # the plans a B200 context uses are the context-free ones
        assert meta["plans"] == {str(k): v for k, v in T.pipeline_plans([S, S_SOFT], knobs).items()}
    changes_plan = "MBE_B200_CHUNKS" in knobs or "MBE_B200_TAPER" in knobs
    assert (meta["plans"][str(S)] != case["default_plans"][S]) == changes_plan, meta["plans"]
    print("\n%s  plan(%d) = %s\n%s" % (name, S, meta["plans"][str(S)], log))
    for c in meta["calls"]:
        lo, hi = _expected_launches(c, meta, knobs)
        if not lo <= c["launches"] <= hi or (meta["kernel_path"] == 1 and (c["launches"] - c["indexed"]) % 3):
            failures.append("%s, %d x %d frames: %d launches, expected %d..%d" % (c["row"], c["n"], c["frames"],
                                                                                c["launches"], lo, hi))

    want = case["want"]
    for row, key, bits in (("host3", "w3", True), ("dev3", "w3", True), ("submit3", "w3", True), ("packed3", "w3", True),
                           ("host0", "w0", True), ("soft0", "ws", True), ("data3", "w3", False), ("datadev3", "w3", False)):
        w = want[key]
        for k in ("pcm", "pcmf", "results") + (("bits",) if bits else ()):
            _diff(failures, row + " " + k, z[row + "." + k], w[k])
        _diff(failures, row + " state", z[row + ".state"], w["state"])
        _diff(failures, row + " rng", z[row + ".rng"], w["rng"])

    ok = case["accepted"]
    w = want["w3"]
    for row in ("idx3", "idxdev3"):
        got = {k: z[row + "." + k] for k in ("pcm", "pcmf", "results", "bits")}
        for k in got:
            _diff(failures, row + " " + k, got[k][ok], w[k][ok])
        # rejected elements: status -1, every other field zero, no PCM and no bits
        res = got["results"][~ok]
        _diff(failures, row + " rejected status", res[..., 0], np.full(res.shape[:-1], -1, np.int32))
        _diff(failures, row + " rejected result fields", res[..., 1:], np.zeros_like(res[..., 1:]))
        for k in ("pcm", "pcmf", "bits"):
            _diff(failures, row + " rejected " + k, got[k][~ok], np.zeros_like(got[k][~ok]))
        _diff(failures, row + " state", z[row + ".state"], w["state"][ok])
        _diff(failures, row + " rng", z[row + ".rng"], w["rng"][ok])
        # the slots no accepted element names keep their state
        _diff(failures, row + " idle state", z[row + ".idle_state_after"], z[row + ".idle_state_before"])
        _diff(failures, row + " idle rng", z[row + ".idle_rng_after"], z[row + ".idle_rng_before"])
    z.close()
    os.remove(out)
    assert not failures, "%s:\n  %s" % (name, "\n  ".join(failures))
