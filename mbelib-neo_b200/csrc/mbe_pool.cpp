// Many GPUs from one process (SURVEY 8(e)): a pool of per-GPU contexts that shards the global stream range into
// contiguous blocks, one block per device, and runs a batched call on every device that owns part of it, concurrently,
// from one host thread per device.  Streams are independent, so nothing is exchanged between GPUs: the host only
// scatters the input bit buffers and gathers PCM / results (plain pointer offsets into the caller's arrays).
// Host-only C++ on top of the C-ABI of include/mbe_b200.h; no CUDA headers.
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <thread>
#include <vector>

#include "../../include/mbe_b200.h"

struct mbe_b200_pool {
    std::vector<mbe_b200_ctx*> ctx;
    std::vector<int> first;   // global id of the first stream of each shard (+ one past the end)
    int max_streams;
    // indexed calls: per shard, a pinned staging buffer (mbe_b200_host_alloc, grown on demand) its elements are gathered into
    std::vector<void*> stage;
    std::vector<size_t> stage_cap;
    char err[320];
};

static char g_pool_err[320] = "";

extern "C" {

int mbe_b200_pool_create(mbe_b200_pool** out, int n_devices, const int* device_ordinals, int max_streams) {
    if (!out || n_devices < 0 || max_streams <= 0) {
        snprintf(g_pool_err, sizeof(g_pool_err), "mbe_b200_pool_create: bad argument");
        return MBE_B200_E_ARG;
    }
    *out = nullptr;
    if (n_devices == 0) {
        n_devices = mbe_b200_device_count();
        device_ordinals = nullptr;
        if (n_devices <= 0) {
            snprintf(g_pool_err, sizeof(g_pool_err), "mbe_b200_pool_create: no CUDA device (there is no CPU fallback)");
            return MBE_B200_E_NOGPU;
        }
    }
    n_devices = std::min(n_devices, max_streams);
    mbe_b200_pool* p = new mbe_b200_pool();
    p->max_streams = max_streams;
    p->err[0] = 0;
    // base + remainder, like sharding.shard_range: n_devices <= max_streams, so no shard is empty and every entry of
    // p->ctx is a live context (9 streams on 8 GPUs: 2 1 1 1 1 1 1 1, not 2 2 2 2 1 0 0 0)
    const int base = max_streams / n_devices, rem = max_streams % n_devices;
    for (int i = 0; i < n_devices; ++i) {
        const int lo = i * base + std::min(i, rem), hi = lo + base + (i < rem ? 1 : 0);
        p->first.push_back(lo);
        mbe_b200_ctx* c = nullptr;
        const int rc = mbe_b200_create(&c, device_ordinals ? device_ordinals[i] : i, hi - lo);
        if (rc != 0) {
            snprintf(g_pool_err, sizeof(g_pool_err), "mbe_b200_pool_create: shard %d: %s", i, mbe_b200_last_error(nullptr));
            for (mbe_b200_ctx* q : p->ctx) {
                mbe_b200_destroy(q);
            }
            delete p;
            return rc;
        }
        p->ctx.push_back(c);
    }
    p->first.push_back(max_streams);
    p->stage.assign(p->ctx.size(), nullptr);
    p->stage_cap.assign(p->ctx.size(), 0);
    *out = p;
    return 0;
}

void mbe_b200_pool_destroy(mbe_b200_pool* p) {
    if (!p) {
        return;
    }
    for (mbe_b200_ctx* c : p->ctx) {
        mbe_b200_destroy(c);
    }
    for (void* b : p->stage) {
        if (b) {
            mbe_b200_host_free(b);
        }
    }
    delete p;
}

const char* mbe_b200_pool_last_error(const mbe_b200_pool* p) { return p ? p->err : g_pool_err; }

int mbe_b200_pool_shards(const mbe_b200_pool* p) { return p ? (int)p->ctx.size() : 0; }

int mbe_b200_pool_shard(const mbe_b200_pool* p, int shard, int* first_stream, int* n_streams, mbe_b200_ctx** ctx) {
    if (!p || shard < 0 || shard >= (int)p->ctx.size()) {
        return MBE_B200_E_ARG;
    }
    if (first_stream) {
        *first_stream = p->first[shard];
    }
    if (n_streams) {
        *n_streams = p->first[shard + 1] - p->first[shard];
    }
    if (ctx) {
        *ctx = p->ctx[shard];
    }
    return 0;
}

}  // extern "C"

// run fn(shard, ctx, local first stream, count, offset of that block inside the caller's range) on every shard that
// overlaps [first, first + count), one host thread per shard; the first failure wins
template <class F>
static int for_each_shard(mbe_b200_pool* p, const char* what, int first, int count, F fn) {
    if (!p) {
        return MBE_B200_E_ARG;
    }
    if (first < 0 || count < 0 || first > p->max_streams - count) {
        snprintf(p->err, sizeof(p->err), "%s: stream range out of bounds", what);
        return MBE_B200_E_ARG;
    }
    const int n = (int)p->ctx.size();
    std::vector<int> rc(n, 0);
    std::vector<std::thread> th;
    for (int i = 0; i < n; ++i) {
        const int lo = std::max(first, p->first[i]), hi = std::min(first + count, p->first[i + 1]);
        if (hi <= lo || !p->ctx[i]) {
            continue;
        }
        th.emplace_back([=, &rc]() { rc[i] = fn(i, p->ctx[i], lo - p->first[i], hi - lo, (size_t)(lo - first)); });
    }
    for (std::thread& t : th) {
        t.join();
    }
    for (int i = 0; i < n; ++i) {
        if (rc[i] != 0) {
            snprintf(p->err, sizeof(p->err), "%s: shard %d: %s", what, i, mbe_b200_last_error(p->ctx[i]));
            return rc[i];
        }
    }
    return 0;
}

extern "C" {

int mbe_b200_pool_init_streams(mbe_b200_pool* p, int first_stream, int count, const uint32_t* seeds) {
    return for_each_shard(p, "pool_init_streams", first_stream, count,
                          [=](int, mbe_b200_ctx* c, int lo, int n, size_t off) {
                              return mbe_b200_init_streams(c, lo, n, seeds ? seeds + off : nullptr);
                          });
}

int mbe_b200_pool_export_state(mbe_b200_pool* p, int first_stream, int count, void* parms_triplets) {
    return for_each_shard(p, "pool_export_state", first_stream, count,
                          [=](int, mbe_b200_ctx* c, int lo, int n, size_t off) {
                              return mbe_b200_export_state(c, lo, n, (uint8_t*)parms_triplets + off * 3 * MBE_B200_PARMS_BYTES);
                          });
}

int mbe_b200_pool_import_state(mbe_b200_pool* p, int first_stream, int count, const void* parms_triplets) {
    return for_each_shard(p, "pool_import_state", first_stream, count,
                          [=](int, mbe_b200_ctx* c, int lo, int n, size_t off) {
                              return mbe_b200_import_state(c, lo, n,
                                                           (const uint8_t*)parms_triplets + off * 3 * MBE_B200_PARMS_BYTES);
                          });
}

// packed < 0: one byte per bit (soft = 0) or mbe_soft_bit pairs (soft = 1); packed = 1: eight hard bits per byte
static int pool_process(mbe_b200_pool* p, const char* what, int codec, int soft, int packed, int first_stream, int n_streams,
                        int n_frames, const uint8_t* frames, int16_t* pcm, float* pcmf, mbe_b200_result* results,
                        uint8_t* bits) {
    int fbits = 0, pbits = 0;
    if (p && (mbe_b200_geometry(codec, &fbits, &pbits) != 0 || n_frames < 0 || !frames)) {
        snprintf(p->err, sizeof(p->err), "%s: bad argument", what);
        return MBE_B200_E_ARG;
    }
    const size_t fbytes = packed ? (size_t)mbe_b200_channel_frame_bytes(p ? p->ctx[0] : nullptr, codec)
                                 : (size_t)fbits * (soft ? 2u : 1u);
    const size_t F = (size_t)n_frames;
    return for_each_shard(p, what, first_stream, n_streams, [=](int, mbe_b200_ctx* c, int lo, int n, size_t off) {
        const uint8_t* fr = frames + off * F * fbytes;
        int16_t* o16 = pcm ? pcm + off * F * MBE_B200_SAMPLES_PER_FRAME : nullptr;
        float* of = pcmf ? pcmf + off * F * MBE_B200_SAMPLES_PER_FRAME : nullptr;
        mbe_b200_result* r = results ? results + off * F : nullptr;
        uint8_t* b = bits ? bits + off * F * (size_t)pbits : nullptr;
        return packed ? mbe_b200_process_frames_packed(c, codec, lo, n, n_frames, fr, o16, of, r, b)
                      : mbe_b200_process_frames(c, codec, soft, lo, n, n_frames, fr, o16, of, r, b);
    });
}

int mbe_b200_pool_set_channel_map(mbe_b200_pool* p, int codec, const uint16_t* map, int n_bits) {
    if (!p) {
        return MBE_B200_E_ARG;
    }
    for (size_t i = 0; i < p->ctx.size(); ++i) {
        if (!p->ctx[i]) {
            continue;
        }
        const int rc = mbe_b200_set_channel_map(p->ctx[i], codec, map, n_bits);
        if (rc != 0) {
            snprintf(p->err, sizeof(p->err), "pool_set_channel_map: shard %d: %s", (int)i, mbe_b200_last_error(p->ctx[i]));
            return rc;
        }
    }
    return 0;
}

int mbe_b200_pool_process_frames(mbe_b200_pool* p, int codec, int soft, int first_stream, int n_streams, int n_frames,
                                 const uint8_t* frames, int16_t* pcm, float* pcmf, mbe_b200_result* results, uint8_t* bits) {
    return pool_process(p, "pool_process_frames", codec, soft ? 1 : 0, 0, first_stream, n_streams, n_frames, frames, pcm, pcmf,
                        results, bits);
}

int mbe_b200_pool_process_frames_packed(mbe_b200_pool* p, int codec, int first_stream, int n_streams, int n_frames,
                                        const uint8_t* packed, int16_t* pcm, float* pcmf, mbe_b200_result* results,
                                        uint8_t* bits) {
    return pool_process(p, "pool_process_frames_packed", codec, 0, 1, first_stream, n_streams, n_frames, packed, pcm, pcmf,
                        results, bits);
}

}  // extern "C"

// ---- indexed calls -----------------------------------------------------------------------------------------------------
// shard owning global slot `slot` (in range)
static int shard_of(const mbe_b200_pool* p, int slot) {
    return (int)(std::upper_bound(p->first.begin(), p->first.end(), slot) - p->first.begin()) - 1;
}

// run fn(shard, ctx, element positions of that shard) on every shard that owns an element, one host thread per shard
template <class F>
static int for_each_part(mbe_b200_pool* p, const char* what, const std::vector<std::vector<int>>& part, F fn) {
    const int n = (int)p->ctx.size();
    std::vector<int> rc(n, 0);
    std::vector<std::thread> th;
    for (int i = 0; i < n; ++i) {
        if (!part[i].empty()) {
            th.emplace_back([&, i]() { rc[i] = fn(i, p->ctx[i], part[i]); });
        }
    }
    for (std::thread& t : th) {
        t.join();
    }
    for (int i = 0; i < n; ++i) {
        if (rc[i] != 0) {
            snprintf(p->err, sizeof(p->err), "%s: shard %d: %s", what, i, mbe_b200_last_error(p->ctx[i]));
            return rc[i];
        }
    }
    return 0;
}

static int grow_stage(mbe_b200_pool* p, int shard, size_t bytes) {
    if (bytes <= p->stage_cap[shard]) {
        return 0;
    }
    if (p->stage[shard]) {
        mbe_b200_host_free(p->stage[shard]);
        p->stage[shard] = nullptr;
        p->stage_cap[shard] = 0;
    }
    const int rc = mbe_b200_host_alloc(&p->stage[shard], bytes);
    if (rc == 0) {
        p->stage_cap[shard] = bytes;
    }
    return rc;
}

static size_t align64(size_t x) { return (x + 63) & ~(size_t)63; }

// One per-element array of an indexed pool call, `bytes` per element (all its frames): `in` arrays are gathered into the
// shard's staging buffer before the context call, `out` arrays scattered back after it (results_inout is both).
// host == nullptr: the array is not used and the context call gets nullptr.
struct IndexedArray {
    uint8_t* host;
    size_t bytes;
    bool in, out;
};

// The shared body of the indexed pool calls.  A stable partition of the element positions by owning shard: a slot always
// maps to one shard, so the context's first-occurrence rule holds for the whole list.  An out-of-range element is rejected
// here as a context rejects it: its output-only arrays are zeroed and the status of each of its `results` frames is set to
// -1 (a frame call's results are output-only and so read zero otherwise, a data call's IN/OUT results keep the caller's
// input).  Every shard then gathers its elements in list order into its pinned staging buffer (local slots first), runs
// call(ctx, local slots, count, local arrays) and scatters the outputs back.
template <class Call>
static int pool_indexed(mbe_b200_pool* p, const char* what, const int32_t* slots, int n, size_t n_frames,
                        mbe_b200_result* results, std::vector<IndexedArray> arr, Call call) {
    std::vector<std::vector<int>> part(p->ctx.size());
    for (int i = 0; i < n; ++i) {
        const int slot = slots[i];
        if (slot >= 0 && slot < p->max_streams) {
            part[shard_of(p, slot)].push_back(i);
            continue;
        }
        for (const IndexedArray& a : arr) {
            if (a.host && !a.in) {
                memset(a.host + (size_t)i * a.bytes, 0, a.bytes);
            }
        }
        for (size_t f = 0; results && f < n_frames; ++f) {
            results[(size_t)i * n_frames + f].status = -1;   // MBE_STATUS_INVALID_ARGUMENT
        }
    }
    return for_each_part(p, what, part, [&](int shard, mbe_b200_ctx* c, const std::vector<int>& el) {
        const size_t m = el.size();
        std::vector<size_t> off(arr.size());
        size_t total = align64(m * sizeof(int32_t));
        for (size_t j = 0; j < arr.size(); ++j) {
            off[j] = total;
            total += arr[j].host ? align64(m * arr[j].bytes) : 0;
        }
        int rc = grow_stage(p, shard, total);
        if (rc != 0) {
            return rc;
        }
        uint8_t* base = (uint8_t*)p->stage[shard];
        int32_t* l_slots = (int32_t*)base;
        std::vector<uint8_t*> local(arr.size());
        for (size_t j = 0; j < arr.size(); ++j) {
            local[j] = arr[j].host ? base + off[j] : nullptr;
        }
        const int lo = p->first[shard];
        for (size_t k = 0; k < m; ++k) {
            l_slots[k] = slots[el[k]] - lo;
            for (size_t j = 0; j < arr.size(); ++j) {
                if (local[j] && arr[j].in) {
                    memcpy(local[j] + k * arr[j].bytes, arr[j].host + (size_t)el[k] * arr[j].bytes, arr[j].bytes);
                }
            }
        }
        rc = call(c, l_slots, (int)m, local.data());
        if (rc != 0) {
            return rc;
        }
        for (size_t k = 0; k < m; ++k) {
            for (size_t j = 0; j < arr.size(); ++j) {
                if (local[j] && arr[j].out) {
                    memcpy(arr[j].host + (size_t)el[k] * arr[j].bytes, local[j] + k * arr[j].bytes, arr[j].bytes);
                }
            }
        }
        return 0;
    });
}

extern "C" {

int mbe_b200_pool_process_indexed(mbe_b200_pool* p, int codec, int input, const int32_t* slots, int n, int n_frames,
                                  const uint8_t* in, int16_t* pcm, float* pcmf, mbe_b200_result* results, uint8_t* bits) {
    if (!p) {
        return MBE_B200_E_ARG;
    }
    int fbits = 0, pbits = 0;
    if (mbe_b200_geometry(codec, &fbits, &pbits) != 0 || input < MBE_B200_INPUT_HARD || input > MBE_B200_INPUT_PACKED ||
        n < 0 || n_frames < 0 || (n > 0 && !slots) || !in) {
        snprintf(p->err, sizeof(p->err), "pool_process_indexed: bad argument");
        return MBE_B200_E_ARG;
    }
    if (n == 0 || n_frames == 0) {
        return 0;
    }
    const size_t F = (size_t)n_frames, NS = MBE_B200_SAMPLES_PER_FRAME;
    const size_t fbytes = input == MBE_B200_INPUT_PACKED ? (size_t)mbe_b200_channel_frame_bytes(p->ctx[0], codec)
                                                         : (size_t)fbits * (input == MBE_B200_INPUT_SOFT ? 2u : 1u);
    return pool_indexed(p, "pool_process_indexed", slots, n, F, results,
                        {{(uint8_t*)in, F * fbytes, true, false},
                         {(uint8_t*)pcm, F * NS * sizeof(int16_t), false, true},
                         {(uint8_t*)pcmf, F * NS * sizeof(float), false, true},
                         {(uint8_t*)results, F * sizeof(mbe_b200_result), false, true},
                         {bits, F * (size_t)pbits, false, true}},
                        [&](mbe_b200_ctx* c, const int32_t* l_slots, int m, uint8_t* const* l) {
                            return mbe_b200_process_indexed(c, codec, input, l_slots, m, n_frames, l[0], (int16_t*)l[1],
                                                            (float*)l[2], (mbe_b200_result*)l[3], l[4]);
                        });
}

int mbe_b200_pool_process_data_indexed(mbe_b200_pool* p, int codec, int packed, const int32_t* slots, int n, int n_frames,
                                       const uint8_t* bits, mbe_b200_result* results_inout, int16_t* pcm, float* pcmf) {
    if (!p) {
        return MBE_B200_E_ARG;
    }
    int fbits = 0, pbits = 0;
    if (mbe_b200_geometry(codec, &fbits, &pbits) != 0 || packed < 0 || packed > 1 || n < 0 || n_frames < 0 ||
        (n > 0 && !slots) || !bits) {
        snprintf(p->err, sizeof(p->err), "pool_process_data_indexed: bad argument");
        return MBE_B200_E_ARG;
    }
    if (n == 0 || n_frames == 0) {
        return 0;
    }
    const size_t F = (size_t)n_frames, NS = MBE_B200_SAMPLES_PER_FRAME;
    const size_t bbytes = packed ? (size_t)mbe_b200_packed_param_bytes(codec) : (size_t)pbits;
    return pool_indexed(p, "pool_process_data_indexed", slots, n, F, results_inout,
                        {{(uint8_t*)bits, F * bbytes, true, false},
                         {(uint8_t*)results_inout, F * sizeof(mbe_b200_result), true, true},
                         {(uint8_t*)pcm, F * NS * sizeof(int16_t), false, true},
                         {(uint8_t*)pcmf, F * NS * sizeof(float), false, true}},
                        [&](mbe_b200_ctx* c, const int32_t* l_slots, int m, uint8_t* const* l) {
                            return mbe_b200_process_data_indexed(c, codec, packed, l_slots, m, n_frames, l[0],
                                                                 (mbe_b200_result*)l[1], (int16_t*)l[2], (float*)l[3]);
                        });
}

int mbe_b200_pool_init_streams_indexed(mbe_b200_pool* p, const int32_t* slots, int n, const uint32_t* seeds) {
    if (!p) {
        return MBE_B200_E_ARG;
    }
    if (n < 0 || (n > 0 && !slots)) {
        snprintf(p->err, sizeof(p->err), "pool_init_streams_indexed: bad argument");
        return MBE_B200_E_ARG;
    }
    std::vector<unsigned char> seen(n > 0 ? (size_t)p->max_streams : 0, 0);
    std::vector<std::vector<int>> part(p->ctx.size());
    for (int i = 0; i < n; ++i) {
        const int slot = slots[i];
        if (slot < 0 || slot >= p->max_streams || seen[slot]) {
            snprintf(p->err, sizeof(p->err), "pool_init_streams_indexed: a slot is outside the pool or listed twice");
            return MBE_B200_E_ARG;
        }
        seen[slot] = 1;
        part[shard_of(p, slot)].push_back(i);
    }
    return for_each_part(p, "pool_init_streams_indexed", part, [&](int shard, mbe_b200_ctx* c, const std::vector<int>& el) {
        std::vector<int32_t> l_slots(el.size());
        std::vector<uint32_t> l_seeds(seeds ? el.size() : 0);
        for (size_t k = 0; k < el.size(); ++k) {
            l_slots[k] = slots[el[k]] - p->first[shard];
            if (seeds) {
                l_seeds[k] = seeds[el[k]];
            }
        }
        return mbe_b200_init_streams_indexed(c, l_slots.data(), (int)el.size(), seeds ? l_seeds.data() : nullptr);
    });
}

}  // extern "C"
