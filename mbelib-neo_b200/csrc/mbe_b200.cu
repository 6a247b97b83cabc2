// libmbe_b200.so - B200 (sm_100a) batched IMBE/AMBE decoder: stream kernels, per-frame state machines,
// host-side context and the C-ABI declared in include/mbe_b200.h.
//
// Execution model: one warp owns one voice stream for the whole launch and walks its frames in order
// (inter-frame prediction, oscillator phases, WOLA tail and noise generator make frames of a stream
// strictly sequential); the three mbe_parms structs of the stream stay in shared memory between
// frames and touch HBM once per launch.  Parallelism is streams x (harmonics | samples | codewords).
// The stream kernel is a template over (codec, soft, mode): every instantiation carries only its own
// front-end, parameter decoder and state machine, so the code a warp walks per frame stays small
// (the first version was one 767 KB kernel and spent 64 % of its stall samples waiting for
// instruction fetch - profiles/r01a_*).
// No tensor cores (no dense contraction in this path), no collectives (streams are independent).
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <mutex>
#include <vector>

#include "mbe_common.cuh"

// ---- codec tables: device copy + host copy (host copy is only used to derive DevTables) ----------
#define MBE_TBL __device__ const
#include "mbe_tables.inc"
#undef MBE_TBL
#define MBE_EXP2_TAB_QUAL __device__ const
#include "mbe_exp2_tab.inc"
#define d_exp2_tab mbe_exp2_tab
namespace hosttab {
#define MBE_TBL static const
#include "mbe_tables.inc"
#undef MBE_TBL
}  // namespace hosttab

#include "mbe_frontend.cuh"
#include "mbe_parms.cuh"
#include "mbe_synth.cuh"
#include "mbe_split.cuh"

#ifndef MBE_SPLIT_DEFAULT
#define MBE_SPLIT_DEFAULT 1
#endif
#ifndef MBE_TOP_BARRIER
#define MBE_TOP_BARRIER 1
#endif
// block barriers between the per-warp stages of a frame (bit mask; see MBE_STAGE_BARRIER in the stream kernel)
#ifndef MBE_BARRIERS
#define MBE_BARRIERS 3
#endif
#define MBE_STAGE_BARRIER(bit) do { if (MBE_BARRIERS & (bit)) __syncthreads(); } while (0)

namespace mbe {

constexpr unsigned FLAG_SOFT = 0x0001u, FLAG_C0 = 0x0002u, FLAG_C4 = 0x0004u, FLAG_TONE = 0x0010u,
                   FLAG_ERASURE = 0x0020u, FLAG_REPEAT = 0x0040u, FLAG_MUTE = 0x0080u;
constexpr unsigned CONTEXT_FLAGS = FLAG_SOFT | FLAG_C0 | FLAG_C4;
constexpr unsigned STATUS_FLAGS = FLAG_TONE | FLAG_ERASURE | FLAG_REPEAT | FLAG_MUTE;

struct FrameCtx {
    int total, c0, c0v, c4, c4v;
    unsigned flags;  // context flags in, status flags accumulate
};

// What the frame's state machine decided to render; executed by ONE shared tail (render_frame) so that
// the synthesis code exists once per kernel.
enum { ACT_VOICE = 0, ACT_REPLAY, ACT_COMFORT_INIT, ACT_COMFORT_ERASURE, ACT_TONE };
struct Action {
    int kind;
    float f1, f2;
    int amp;
    int keep_prev;  // ACT_TONE: prev_mp <- cur_mp afterwards (D-STAR clean tone)
};

// src/internal/mbe_result.h:44-97
__device__ __forceinline__ int resolve_total_errors(int c0, int prot, int c4, int total_in, unsigned flags, int* total) {
    auto ok = [](int c) { return c >= 0 && c <= 184; };
    if ((flags & ~(CONTEXT_FLAGS | STATUS_FLAGS)) != 0u) {
        return -1;
    }
    if (!ok(c0) || !ok(prot) || !ok(c4) || !ok(total_in)) {
        return -1;
    }
    if (c0 > 184 - prot) {
        return -1;
    }
    const int comp = c0 + prot;
    if (!ok(comp)) {
        return -1;
    }
    const int t = (total_in == 0 && comp != 0) ? comp : total_in;
    const bool c0v = (flags & FLAG_C0) != 0u, c4v = (flags & FLAG_C4) != 0u;
    if (!((comp == 0 || t == comp) && (!c0v || t >= c0) && (!c4v || t >= c4))) {
        return -1;
    }
    *total = t;
    return 0;
}

// ---- IMBE 4400 frame state machine (imbe7200x4400.c:780-888) --------------------------------------
template <class H>
__device__ __forceinline__ Action process_imbe(FrameCtx& fc, const unsigned dw[3], WarpWS& ws, const H& home,
                                               const DevTables* T, int lane) {
    ParmsSmall& cur = ws.cur;
    PrevSmall& prev = ws.prev;
    const float rate = (0.95f * prev.errorRate) + (0.000365f * (float)fc.total);
    __syncwarp();
    if (lane == 0) {
        cur.errorCount4 = fc.c4v ? fc.c4 : 0;
        cur.mutingThreshold = 0.0875f;
        cur.errorCountTotal = fc.total;
        cur.errorRate = rate;
    }
    __syncwarp();
    const int bad = decode_imbe(dw, ws, T, lane);
    __syncwarp();
    const float thr = 10.0f + (40.0f * rate);
    bool repeat;
    if (bad == 1) {
        repeat = true;
    } else if (fc.c0v) {
        repeat = (fc.c0 >= 2) && ((float)fc.total >= thr);
    } else {
        repeat = fc.total > 5;
    }
    if (!repeat) {
        if (lane == 0) {
            cur.repeatCount = 0;
        }
    } else {
        if (prev.repeatCount > 3) {
            // headroom exhausted: default voice model, continuity state kept (imbe7200x4400.c:56-81)
            for (int l = lane; l <= 56; l += 32) {
                cur.Vl[l] = 0;
                cur.Ml[l] = 1.0f;
                cur.log2Ml[l] = 0.0f;
            }
            if (lane == 0) {
                cur.swn = 0;
                cur.tonePhase = 0;
                cur.w0 = T->imbe_default_w0;
                ws.w0row = COSW_IMBE_DEFAULT;
                cur.L = T->imbe_default_L;
                cur.K = 12;
                cur.gamma = 0.0f;
                cur.repeatCount = 0;
                cur.localEnergy = 75000.0f;
                cur.amplitudeThreshold = 20480;
                cur.mutingThreshold = 0.0875f;
            }
        } else {
            cur_from_prev(ws, home, lane);
            if (lane == 0) {
                cur.repeatCount = cur.repeatCount + 1;
            }
        }
        fc.flags |= FLAG_REPEAT;
    }
    __syncwarp();
    if ((cur.repeatCount >= 4) || (cur.errorRate > cur.mutingThreshold)) {
        fc.flags |= FLAG_MUTE;
    }
    Action a = {ACT_VOICE, 0.0f, 0.0f, 0, 0};
    return a;
}

// ---- AMBE helpers (ambe_common.c:191-271) ----------------------------------------------------------
template <class H>
__device__ __forceinline__ void init_ambe(WarpWS& ws, const H& home, const DevTables* T, int lane) {
    init_all(ws, home, T->ambe_default_w0, 15, 0, 0.096f, lane);
}

// erasure model built in cur_mp from prev_mp: phases, noise generator and WOLA tail carried over
template <class H>
__device__ __forceinline__ void set_erasure_model(WarpWS& ws, const H& home, int lane) {
    ParmsSmall& mp = ws.cur;
    const PrevSmall& src = ws.prev;
    __syncwarp();
    for (int l = lane; l <= 56; l += 32) {
        mp.Ml[l] = 1.0f;
        mp.Vl[l] = 0;
        mp.log2Ml[l] = 0.0f;
        // prev_mp's phases live in its HBM image (PHIl at words 174.., PSIl at 231..), PHIl[0] in shared memory
        mp.PHIl[l] = (l == 0) ? src.PHIl0 : __uint_as_float(home.prev[174 + l]);
        mp.PSIl[l] = __uint_as_float(home.prev[231 + l]);
    }
    bulk_copy(ws, home, home.cur, home.prev, OP_CUR_FROM_PREV, lane);
    if (lane == 0) {
        mp.swn = 0;
        mp.tonePhase = 0;
        mp.w0 = 0.0f;
        mp.L = 9;
        mp.K = 0;
        mp.gamma = 0.0f;
        mp.localEnergy = 75000.0f;
        mp.amplitudeThreshold = 20480;
        mp.noiseSeed = src.noiseSeed;
    }
    __syncwarp();
}

template <class H>
__device__ __forceinline__ void prepare_ambe(const FrameCtx& fc, WarpWS& ws, const H& home, const DevTables* T,
                                             int lane) {
    if (fabsf(ws.prev.mutingThreshold - 0.096f) > 1e-6f) {
        __syncwarp();
        init_ambe(ws, home, T, lane);  // first AMBE frame after a generic init
    }
    const float rate = (0.95f * ws.prev.errorRate) + (0.001064f * (float)fc.total);
    __syncwarp();
    if (lane == 0) {
        ws.cur.mutingThreshold = 0.096f;
        ws.cur.errorCountTotal = fc.total;
        ws.cur.errorCount4 = 0;
        ws.cur.errorRate = rate;
    }
    __syncwarp();
}

__device__ __forceinline__ int ambe_voice_or_mute(FrameCtx& fc, const WarpWS& ws) {
    if (ws.cur.repeatCount < 4) {
        return ACT_VOICE;
    }
    fc.flags |= FLAG_MUTE;
    return ACT_COMFORT_INIT;
}

template <class H>
__device__ __forceinline__ void ambe_repeat(WarpWS& ws, const H& home, FrameCtx& fc, int lane) {
    cur_from_prev(ws, home, lane);
    if (lane == 0) {
        ws.cur.repeatCount = ws.cur.repeatCount + 1;
    }
    fc.flags |= FLAG_REPEAT;
    __syncwarp();
}

// ---- AMBE+2 3600x2450 (ambe3600x2450.c:716-877) -----------------------------------------------------
template <class H>
__device__ __forceinline__ Action process_ambe2450(FrameCtx& fc, const unsigned dw[3], WarpWS& ws,
                                                   const H& home, const DevTables* T, int lane) {
    Action act = {ACT_COMFORT_INIT, 0.0f, 0.0f, 0, 0};
    prepare_ambe(fc, ws, home, T, lane);
    const int bad = decode_ambe2450(dw, ws, T, fc.total, lane);
    __syncwarp();
    if (bad == 2) {
        fc.flags |= FLAG_ERASURE;
        if (lane == 0) {
            ws.cur.repeatCount = 0;
        }
        set_erasure_model(ws, home, lane);
    } else if (bad == 7) {
        fc.flags |= FLAG_TONE;
        if (lane == 0) {
            ws.cur.repeatCount = 0;
        }
    } else {
        const bool repeat = fc.c0v ? ((fc.c0 >= 4) || ((fc.c0 >= 2) && (fc.total >= 6))) : (fc.total > 3);
        if (repeat) {
            ambe_repeat(ws, home, fc, lane);
        } else if (lane == 0) {
            ws.cur.repeatCount = 0;
        }
    }
    __syncwarp();

    if (bad == 0) {
        act.kind = ambe_voice_or_mute(fc, ws);
    } else if (bad == 7) {
        unsigned u0 = 0, u1 = 0, u3 = 0;
        for (int i = 0; i < 12; ++i) {
            u0 = (u0 << 1) | getbit(dw, i);
        }
        for (int i = 12; i < 24; ++i) {
            u1 = (u1 << 1) | getbit(dw, i);
        }
        for (int i = 35; i < 49; ++i) {
            u3 = (u3 << 1) | getbit(dw, i);
        }
        const int id1 = (int)((u1 & 0xfffu) >> 4);
        if (tone_freqs(id1, &act.f1, &act.f2)) {
            act.kind = ACT_TONE;
            act.amp = (int)(((u0 & 0x3fu) << 1) + ((u3 >> 4) & 1u));
        } else if (!(ws.prev.repeatCount >= 4)) {
            // invalid tone id: replay the last voice model while advancing synthesis state
            // (ambe3600x2450.c:808-816)
            act.kind = ACT_REPLAY;
        }
    } else if (bad == 2) {
        act.kind = ACT_COMFORT_ERASURE;
    }
    return act;
}

// ---- AMBE 3600x2400 (ambe3600x2400.c:629-762) --------------------------------------------------------
template <class H>
__device__ __forceinline__ Action process_ambe2400(FrameCtx& fc, const unsigned dw[3], WarpWS& ws,
                                                   const H& home, const DevTables* T, int lane) {
    Action act = {ACT_COMFORT_INIT, 0.0f, 0.0f, 0, 0};
    prepare_ambe(fc, ws, home, T, lane);
    const int bad = decode_ambe2400(dw, ws, T, lane);
    __syncwarp();
    const bool clean_tone = (bad >= 7) && (bad <= 122) && (fc.c0 < 2) && (fc.total < 3);
    if (bad == 3) {
        fc.flags |= FLAG_TONE;
        if (lane == 0) {
            ws.cur.repeatCount = 0;
        }
    } else if (clean_tone) {
        // state untouched
    } else if (fc.total > 3) {
        ambe_repeat(ws, home, fc, lane);
    } else if (lane == 0) {
        ws.cur.repeatCount = 0;
    }
    __syncwarp();

    if (clean_tone) {
        act.kind = ACT_TONE;
        act.f1 = act.f2 = 31.25f * (float)bad;
        act.amp = 103;
        act.keep_prev = 1;
    } else if (bad == 0) {
        act.kind = ambe_voice_or_mute(fc, ws);
    }
    return act;
}

// ---- rendering what the state machine decided ---------------------------------------------------------
// A frame is rendered in three steps so that the voiced bank can be shared by the whole block:
//   render_begin   per warp: non-voice actions completely (tone, comfort noise); for voice frames the
//                  enhance + smoothing + phase + component-list part (imbe7200x4400.c:842-856,
//                  ambe3600x2450.c:785-799).  Returns 1 if the frame goes through the bank.
//   voiced_bank_block  all warps of the block together.
//   render_end     per warp: unvoiced synthesis, clip, state hand-over.
// render_begin is split in two (enhancement | synthesis set-up) and render_end in three (forward transform |
// shaping + backward transform | overlap-add + hand-over) so that the kernel can put block barriers between the
// stages: warps of a block that walk the same code share their instruction fetches.
struct RenderState {
    int voice;      // frame runs the speech synthesiser (ACT_VOICE or ACT_REPLAY)
    int has_rm0;
    float rm0;
};

template <bool AMBE, class H>
__device__ __forceinline__ RenderState render_begin1(const Action& act, WarpWS& ws, const H& home,
                                                     const DevTables* T, int lane) {
    RenderState rs = {0, 0, 0.0f};
    int kind = act.kind;
    if (!AMBE) {
        kind = ACT_VOICE;
    }
    if (kind == ACT_VOICE || kind == ACT_REPLAY) {
        rs.voice = 1;
        if (kind == ACT_VOICE) {
            prev_from_cur(ws, home, lane);
            rs.rm0 = spectral_enhance(ws, T, reinterpret_cast<float*>(&ws.u), lane);
            rs.has_rm0 = 1;
        } else {
            // replay the last voice model (ambe3600x2450.c:808-816): cur_mp is parked in the stream's scratch image
            const uint32_t* cw = reinterpret_cast<const uint32_t*>(&ws.cur);
            for (int i = lane; i < HEAD_WORDS; i += 32) {
                home.spill[i] = cw[i];
            }
            if (lane == 0) {
                home.spill[SEED_WORD] = cw[HEAD_WORDS];
            }
            bulk_copy(ws, home, home.spill, home.cur, OP_SPILL_FROM_CUR, lane);
            __syncwarp();
            cur_from_enh(ws, home, lane);
        }
        return rs;
    }
    if (AMBE) {
        if (kind == ACT_TONE) {
            render_tone(ws, act.f1, act.f2, act.amp, lane);
            if (act.keep_prev) {
                prev_from_cur(ws, home, lane);
            }
            return rs;
        }
        comfort_noise(ws, T, lane);
        if (kind == ACT_COMFORT_ERASURE) {
            prev_from_cur(ws, home, lane);
            enh_from_cur(ws, home, lane);
        } else {
            init_ambe(ws, home, T, lane);
        }
    }
    return rs;
}

template <class H>
__device__ __forceinline__ int render_begin2(const RenderState& rs, WarpWS& ws, const H& home, const DevTables* T,
                                             int lane) {
    if (!rs.voice) {
        return 0;
    }
    return synth_begin<true>(ws, reinterpret_cast<const float*>(home.cur + OVERLAP_WORD), T, rs.has_rm0, rs.rm0, lane);
}

// after the overlap-add: prev_mp_enhanced <- cur_mp, and the replay path puts the parked cur_mp back
template <bool AMBE, class H>
__device__ __forceinline__ void render_end(const Action& act, const RenderState& rs, int go, WarpWS& ws,
                                           const H& home, int lane) {
    if (!rs.voice) {
        return;
    }
    enh_from_cur(ws, home, lane, /*bulk=*/!go);
    if (AMBE && act.kind == ACT_REPLAY) {
        uint32_t* cw = reinterpret_cast<uint32_t*>(&ws.cur);
        for (int i = lane; i < HEAD_WORDS; i += 32) {
            cw[i] = home.spill[i];
        }
        if (lane == 0) {
            cw[HEAD_WORDS] = home.spill[SEED_WORD];  // written by lane 0 above
        }
        bulk_copy(ws, home, home.cur, home.spill, OP_CUR_FROM_SPILL, lane);
        __syncwarp();
    }
}

__device__ __forceinline__ void load_block_tables(BlockTables* bt, const DevTables* T) {
    for (int i = threadIdx.x; i < 2 * NS; i += blockDim.x) {
        bt->voiced_win[i < NS ? i : i + (WIN_PREV - NS)] = T->voiced_win[i];
    }
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        bt->tw[i] = T->tw[i];
        bt->uvwin[i] = T->uvwin[i];
    }
    for (int i = threadIdx.x; i < 160; i += blockDim.x) {
        bt->wola_wp[i] = T->wola_wp[i];
        bt->wola_wc[i] = T->wola_wc[i];
        bt->wola_den[i] = T->wola_den[i];
    }
    if (threadIdx.x < 32) {
        bt->uv_jump[threadIdx.x] = make_uint2(T->uvA[threadIdx.x], T->uvC[threadIdx.x]);
    }
    __syncthreads();
}

__device__ __forceinline__ void store_pcm(const LaunchArgs& A, const WarpWS& ws, size_t frame_idx, int lane) {
    if (MBE_ABL & 256) {
        return;
    }
#pragma unroll
    for (int ch = 0; ch < 5; ++ch) {
        const size_t o = frame_idx * NS + 32 * ch + lane;
        const float v = ws.out[32 * ch + lane];
        if (A.pcmf) {
            A.pcmf[o] = ref_nan(v * A.pcmf_scale);  // x 1.0f is exact: the default is the reference's float scale
        }
        if (A.pcm) {
            A.pcm[o] = float_to_short(v);
        }
    }
}

// stream state: HBM slot <-> shared memory (the three structs without their bulk arrays, which stay in HBM)
// All 23 loads of a lane are issued before the first one is consumed: with one frame per launch (a real-time server)
// the state round trip is a large part of a stream's lifetime, and one load at a time costs ~20 HBM latencies.
__device__ __forceinline__ void load_stream(WarpWS& ws, const uint32_t* gs, int lane) {
    uint32_t* c = reinterpret_cast<uint32_t*>(&ws.cur);
    uint32_t* p = reinterpret_cast<uint32_t*>(&ws.prev);
    uint32_t* e = reinterpret_cast<uint32_t*>(&ws.enh);
    constexpr int NC = (HEAD_WORDS + 31) / 32, NP = (PREV_WORDS + 31) / 32, NE = (ENH_WORDS + 31) / 32;
    uint32_t vc[NC], vp[NP], ve[NE];
#pragma unroll
    for (int k = 0; k < NC; ++k) {
        const int i = lane + 32 * k;
        vc[k] = (i < HEAD_WORDS) ? gs[i] : 0u;
    }
#pragma unroll
    for (int k = 0; k < NP; ++k) {
        const int j = lane + 32 * k;
        vp[k] = (j < PREV_WORDS) ? gs[PARMS_WORDS + prev_word(j)] : 0u;
    }
#pragma unroll
    for (int k = 0; k < NE; ++k) {
        const int j = lane + 32 * k;
        ve[k] = (j < ENH_WORDS) ? gs[2 * PARMS_WORDS + enh_word(j)] : 0u;
    }
    uint32_t r0 = 0, r1 = 0, r2 = 0, r3 = 0, seed = 0;
    if (lane == 0) {
        seed = gs[SEED_WORD];
        r0 = gs[3 * PARMS_WORDS];
        r1 = gs[3 * PARMS_WORDS + 1];
        r2 = gs[3 * PARMS_WORDS + 2];
        r3 = gs[3 * PARMS_WORDS + 3];
    }
#pragma unroll
    for (int k = 0; k < NC; ++k) {
        const int i = lane + 32 * k;
        if (i < HEAD_WORDS) {
            c[i] = vc[k];
        }
    }
#pragma unroll
    for (int k = 0; k < NP; ++k) {
        const int j = lane + 32 * k;
        if (j < PREV_WORDS) {
            p[j] = vp[k];
        }
    }
#pragma unroll
    for (int k = 0; k < NE; ++k) {
        const int j = lane + 32 * k;
        if (j < ENH_WORDS) {
            e[j] = ve[k];
        }
    }
    if (lane == 0) {
        c[HEAD_WORDS] = seed;
        ws.rng.comfort = (unsigned long long)r0 | ((unsigned long long)r1 << 32);
        ws.rng.uv_seed = r2;
        ws.rng.uv_override = r3;
    }
    __syncwarp();
}

__device__ __forceinline__ void store_stream(const WarpWS& ws, uint32_t* gs, int lane) {
    const uint32_t* c = reinterpret_cast<const uint32_t*>(&ws.cur);
    const uint32_t* p = reinterpret_cast<const uint32_t*>(&ws.prev);
    const uint32_t* e = reinterpret_cast<const uint32_t*>(&ws.enh);
    __syncwarp();
    for (int i = lane; i < HEAD_WORDS; i += 32) {
        gs[i] = c[i];
    }
    for (int j = lane; j < PREV_WORDS; j += 32) {
        gs[PARMS_WORDS + prev_word(j)] = p[j];
    }
    for (int j = lane; j < ENH_WORDS; j += 32) {
        gs[2 * PARMS_WORDS + enh_word(j)] = e[j];
    }
    if (lane == 0) {
        gs[SEED_WORD] = c[HEAD_WORDS];
        gs[3 * PARMS_WORDS] = (uint32_t)(ws.rng.comfort & 0xffffffffULL);
        gs[3 * PARMS_WORDS + 1] = (uint32_t)(ws.rng.comfort >> 32);
        gs[3 * PARMS_WORDS + 2] = ws.rng.uv_seed;
        gs[3 * PARMS_WORDS + 3] = ws.rng.uv_override;
    }
}

// =====================================================================================================
// The stream kernel: CODEC in {0..3}, SOFT in {0 hard bytes, 1 soft bits, 2 hard bits packed 8 per byte},
// MODE in {MODE_FRAMES, MODE_DATA}
// One block = WARPS_PER_BLOCK streams walking their frames in lockstep (see WARPS_PER_BLOCK).
// =====================================================================================================
// SPLIT: the parameter kernel of the two-kernel path (mbe_split.cuh): no oscillator bank, no transforms; every frame
// leaves a descriptor for mbe_split_synth_kernel, frames without speech synthesis are finished here.
// block shape of the stream kernel: the multi-kernel path's parameter kernel on hard-decision input has no tile and fits 64
// registers, so it runs P_WARPS warps per block on the short per-warp stride
template <int SOFT, bool SPLIT>
struct StreamShape {
    static constexpr bool SMALL = SPLIT && SOFT != 1;
    static constexpr int WARPS = SMALL ? P_WARPS : WARPS_PER_BLOCK;
    static constexpr size_t STRIDE = SMALL ? WS_STRIDE_SMALL : sizeof(WarpWS);
    static constexpr int MINB = SMALL ? P_MINB : MIN_BLOCKS_PER_SM;
};

// INDEXED: an indexed call (LaunchArgs::slots); a separate image, so that the contiguous launches keep the register
// allocation they have without the slot list and the claim check.  Indexed MODE_DATA launches also take packed parameter
// bits (LaunchArgs::packed_bytes != 0), a warp-uniform run-time choice rather than another image.
template <int CODEC, int SOFT, int MODE, bool SPLIT, bool INDEXED = false>
__global__ void __launch_bounds__(StreamShape<SOFT, SPLIT>::WARPS * 32, StreamShape<SOFT, SPLIT>::MINB)
mbe_stream_kernel(const LaunchArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using Shape = StreamShape<SOFT, SPLIT>;
    BlockTables* bt = reinterpret_cast<BlockTables*>(smem_raw);
    WarpWS* wsa = reinterpret_cast<WarpWS*>(smem_raw + sizeof(BlockTables));
    BlockShared* bs = reinterpret_cast<BlockShared*>(smem_raw + sizeof(BlockTables) + WARPS_PER_BLOCK * sizeof(WarpWS));
    const DevTables* T = A.tab;
    if (!SPLIT && threadIdx.x == 0) {
        bs->n_interp[0] = bs->n_interp[1] = 0;
    }
    load_block_tables(bt, T);   // ends with a block barrier

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int s = blockIdx.x * Shape::WARPS + warp;
    const bool live = s < A.n_streams;  // idle warps of the last block still take part in the bank
    WarpWS& ws = *reinterpret_cast<WarpWS*>(smem_raw + sizeof(BlockTables) + (size_t)warp * Shape::STRIDE);
    constexpr bool AMBE = (CODEC >= MBE_B200_AMBE3600X2400);
    constexpr int fbits = (CODEC == MBE_B200_IMBE7200X4400) ? 184 : (CODEC == MBE_B200_IMBE7100X4400 ? 168 : 96);
    constexpr int pbits = AMBE ? 49 : 88;
    constexpr bool PACKED = (SOFT == 2);
    const bool data_packed = INDEXED && MODE == MODE_DATA && A.packed_bytes != 0;
    const size_t fstride = (MODE == MODE_DATA) ? (data_packed ? (size_t)A.packed_bytes : (size_t)pbits)
                                               : (PACKED ? (size_t)A.packed_bytes : (size_t)fbits * (SOFT == 1 ? 2u : 1u));

    // an element of an indexed call whose slot is out of range or claimed by an earlier element is rejected: it touches no
    // state, runs no decode, and its outputs are those of an invalid-argument frame (status -1, zeros)
    int slot = A.first_stream + (live ? s : 0);   // slot_of(A, s) of a contiguous launch
    bool own = live;
    if (INDEXED && live) {
        slot = slot_of(A, s);
        own = (unsigned)slot < (unsigned)A.max_streams && A.claim[slot] == claim_tag(A.epoch, A.slot_base + A.io_base + s);
        slot = own ? slot : 0;
    }
    uint32_t* gs = A.state + (size_t)slot * STATE_WORDS;
    const StreamHomeT<SPLIT> home = {gs, gs + PARMS_WORDS, gs + 2 * PARMS_WORDS, gs + SPILL_WORD};
    if (own) {
        load_stream(ws, gs, lane);
    }
    if (lane == 0) {
        ws.w0row = ws.w0row_prev = ws.w0row_enh = -1;
        ws.ops = ws.nops = 0;
    }

    StageTimer tm;
#if MBE_STAGE_TIMING
    for (int i = 0; i < 16; ++i) {
        tm.acc[i] = 0;
    }
    tm.last = clock64();
#endif
#pragma unroll 1
    for (int f = 0; f < A.n_frames; ++f) {
        // no barrier at the frame boundary: the bank's last barrier has retired every cross-warp read of the
        // previous frame's tiles and component lists, and the counters are double-buffered by frame parity
#if MBE_TOP_BARRIER
        __syncthreads();  // keeps the block's warps on the same code (instruction-cache locality)
#endif
        STAGE_T(0);

        const size_t idx = (size_t)(A.io_base + s) * A.n_frames + f;   // element of the caller's [stream][frame] arrays
        unsigned dw[3] = {0u, 0u, 0u};
        FrameCtx fc;
        int status = -1, go = 0;
        Action act = {ACT_COMFORT_INIT, 0.0f, 0.0f, 0, 0};
        mbe_b200_result rout;
        rout.c0_errors = rout.protected_errors = rout.c4_errors = rout.total_errors = 0;
        rout.flags = 0;

        if (own) {
            const uint8_t* fr = A.frames + idx * fstride;
            if (MODE == MODE_FRAMES) {
                // soft decision: the parity cost table takes the whole union and the small tables, reliabilities and
                // corrected rows live in the sample row, which is dead until the synthesis writes it
                SoftScratch S = {nullptr, nullptr, nullptr};
                unsigned char* relp = ws.u.dec.rel;
                unsigned* rowp = ws.u.dec.rowbits;
                if (SOFT == 1) {
                    unsigned char* o = reinterpret_cast<unsigned char*>(ws.out);
                    S.cp = reinterpret_cast<unsigned short*>(&ws.u);
                    S.ka = reinterpret_cast<unsigned*>(o);
                    S.qa = reinterpret_cast<unsigned short*>(o + 256);
                    relp = o + 384;
                    rowp = reinterpret_cast<unsigned*>(o + 576);
                }
                FrontResult R = front_end(CODEC, SOFT == 1, PACKED, fr, dw, relp, S, rowp, T, lane);
                status = R.status;
                fc.total = R.c0 + R.prot;
                fc.c0 = R.c0;
                fc.c0v = 1;
                fc.c4 = R.c4;
                fc.c4v = (R.flags & FLAG_C4) ? 1 : 0;
                fc.flags = R.flags;
            } else {
                // parameter bits from memory + optional decode context (mbe_process<Codec>Data semantics)
                bool bad = false;
#pragma unroll
                for (int w = 0; w < 3; ++w) {
                    const int i = 32 * w + lane;
                    unsigned b = 0;
                    if (i < pbits) {
                        // packed: bit i is bit 7 - (i & 7) of byte i >> 3 (MSB first), so it can only be 0 or 1
                        const unsigned v = data_packed ? (fr[i >> 3] >> (7 - (i & 7))) & 1u : fr[i];
                        bad |= (v > 1u);
                        b = v & 1u;
                    }
                    dw[w] = __ballot_sync(FULL, b);
                }
                int c0 = 0, prot = 0, c4 = 0, tin = 0;
                unsigned fl = 0;
                if (A.results) {
                    const mbe_b200_result rin = A.results[idx];
                    c0 = rin.c0_errors;
                    prot = rin.protected_errors;
                    c4 = rin.c4_errors;
                    tin = rin.total_errors;
                    fl = rin.flags;
                    rout = rin;
                }
                int total = 0;
                status = resolve_total_errors(c0, prot, c4, tin, fl, &total);
                if (status == 0 && __any_sync(FULL, bad)) {
                    status = -2;
                }
                fc.flags = fl & CONTEXT_FLAGS;
                fc.c0v = (fl & FLAG_C0) ? 1 : 0;
                fc.c4v = (fl & FLAG_C4) ? 1 : 0;
                fc.c0 = fc.c0v ? c0 : 0;
                fc.c4 = fc.c4v ? c4 : 0;
                fc.total = total;
            }
        } else if (INDEXED && MODE == MODE_DATA && live && A.results) {
            // a rejected element echoes the caller's decode context with only .status replaced, the rule of every
            // negative status on this path (the location is the caller's I/O element, not stream state)
            rout = A.results[idx];
        }
        // ECC front-end | parameter decode: soft-decision kernels re-join here, because their front-end runs a data-dependent
        // number of coset walks per stream and the block would otherwise walk the parameter decode out of step (instruction
        // fetch stalls; +6 to +13 % on soft input, profiles/experiments/r01z_soft_front_end_barrier.txt)
        if (SOFT == 1 && MODE == MODE_FRAMES) {
            __syncthreads();
        } else {
            MBE_STAGE_BARRIER(16);
        }
        if (live) {
            if (status >= 0) {
                if (!AMBE) {
                    act = process_imbe(fc, dw, ws, home, T, lane);
                } else if (CODEC == MBE_B200_AMBE3600X2400) {
                    act = process_ambe2400(fc, dw, ws, home, T, lane);
                } else {
                    act = process_ambe2450(fc, dw, ws, home, T, lane);
                }
                STAGE_T(1);
            }
        }
        RenderState rs = {0, 0, 0.0f};
        MBE_STAGE_BARRIER(1);   // decode | enhancement
        const bool ok = live && status >= 0;
        if (ok) {
            rs = render_begin1<AMBE>(act, ws, home, T, lane);
        } else if (live) {
            zero_out(ws, lane);
        }
        MBE_STAGE_BARRIER(2);   // enhancement | synthesis set-up
        if (ok) {
            go = render_begin2(rs, ws, home, T, lane);
            STAGE_T(2);
        }
        if (SPLIT) {
            if (live) {
                uint32_t* dsc = A.desc + ((size_t)s * A.n_frames + f) * DESC_WORDS;
                float seed_before = 0.0f;
                if (go) {
                    float ov[3];
                    make_noise_state(ws, reinterpret_cast<float*>(home.cur + OVERLAP_WORD),
                                     reinterpret_cast<float*>(home.enh + OVERLAP_WORD), bt, lane, ov, &seed_before);
                    record_op(ws, OP_SYNTH, lane);
                    emit_desc_arrays(dsc, ws, ov, T, lane);
                }
                emit_desc_info(dsc, ws, go, seed_before, lane);
                if (status >= 0) {
                    render_end<AMBE>(act, rs, go, ws, home, lane);
                    STAGE_T(5);
                    status = fc.total;
                    rout.c0_errors = fc.c0;
                    rout.c4_errors = fc.c4;
                    rout.total_errors = fc.total;
                    rout.protected_errors = fc.total - fc.c0;
                    rout.flags = fc.flags;
                }
                __syncwarp();
                emit_desc_ops(dsc, ws, lane);
                if (lane == 0) {
                    ws.ops = ws.nops = 0;
                }
                if (!go) {
                    store_pcm(A, ws, idx, lane);   // silence, tone or comfort noise: complete without the synthesis kernel
                }
            }
        } else {
        publish_components(bs, f & 1, ws, go, warp, lane);
        __syncthreads();
        STAGE_T(3);
        voiced_bank_block(wsa, bs, f & 1, bt, T, tm, warp, lane);
        STAGE_T(4);

        WolaTail tail;
        if (go) {
            synth_finish_a(ws, home.cur, home.enh, T, bt, lane);
        }
        MBE_STAGE_BARRIER(4);   // forward transform | shaping + backward transform
        if (go) {
            tail = synth_finish_b(ws, home.enh, bt, lane);
        }
        MBE_STAGE_BARRIER(8);   // backward transform | overlap-add, hand-over, stores
        if (live) {
            if (status >= 0) {
                if (go) {
                    synth_finish_c(ws, home.cur, home.enh, tail, bt, lane);
                }
                render_end<AMBE>(act, rs, go, ws, home, lane);
                STAGE_T(5);
                status = fc.total;
                rout.c0_errors = fc.c0;
                rout.c4_errors = fc.c4;
                rout.total_errors = fc.total;
                rout.protected_errors = fc.total - fc.c0;
                rout.flags = fc.flags;
            }
            __syncwarp();
            store_pcm(A, ws, idx, lane);
        }
        }
        if (live) {
            if (A.results && lane == 0) {
                rout.status = status;
                A.results[idx] = rout;
            }
            if (A.bits && MODE == MODE_FRAMES) {
#pragma unroll
                for (int w = 0; w < 3; ++w) {
                    const int i = 32 * w + lane;
                    if (i < pbits) {
                        A.bits[idx * pbits + i] = (uint8_t)((dw[w] >> lane) & 1u);
                    }
                }
            }
        }
        STAGE_T(6);
    }
    if (own) {
        store_stream(ws, gs, lane);
    }
#if MBE_STAGE_TIMING
    STAGE_T(7);
    if (A.dbg && lane == 0 && live) {
        for (int i = 0; i < 16; ++i) {
            atomicAdd(reinterpret_cast<unsigned long long*>(A.dbg) + i, (unsigned long long)tm.acc[i]);
        }
    }
#endif
}

// batched mbe_synthesizeSpeech[f]: element s synthesises one frame from parameter blobs in device memory
// (cur[s] -> ws.cur, prev[s] -> ws.enh; prev's previousUw is read in place, both are updated in place)
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32, MIN_BLOCKS_PER_SM) mbe_synth_kernel(const LaunchArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    BlockTables* bt = reinterpret_cast<BlockTables*>(smem_raw);
    WarpWS* wsa = reinterpret_cast<WarpWS*>(smem_raw + sizeof(BlockTables));
    BlockShared* bs = reinterpret_cast<BlockShared*>(smem_raw + sizeof(BlockTables) + WARPS_PER_BLOCK * sizeof(WarpWS));
    const DevTables* T = A.tab;
    load_block_tables(bt, T);
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int s = blockIdx.x * WARPS_PER_BLOCK + warp;
    const bool live = s < A.n_streams;
    WarpWS& ws = wsa[warp];
    uint32_t* gc = A.synth_cur + (size_t)(live ? s : 0) * PARMS_WORDS;
    uint32_t* gp = A.synth_prev + (size_t)(live ? s : 0) * PARMS_WORDS;
    uint32_t* c = reinterpret_cast<uint32_t*>(&ws.cur);
    uint32_t* e = reinterpret_cast<uint32_t*>(&ws.enh);
    int go = 0;
    if (live) {
        for (int i = lane; i < HEAD_WORDS; i += 32) {
            c[i] = gc[i];
        }
        for (int j = lane; j < ENH_WORDS; j += 32) {
            e[j] = gp[enh_word(j)];
        }
        // RNG as after mbe_setThreadRngSeed(seed) (mbelib.c:173-181); no seeds: fresh-thread defaults
        if (lane == 0) {
            ws.w0row = ws.w0row_prev = ws.w0row_enh = -1;
            c[HEAD_WORDS] = gc[SEED_WORD];
            if (A.synth_rng) {  // the caller's RNG words, carried from call to call (single-stream shim)
                const uint32_t* r = A.synth_rng + 4 * (size_t)s;
                ws.rng.comfort = (unsigned long long)r[0] | ((unsigned long long)r[1] << 32);
                ws.rng.uv_seed = r[2];
                ws.rng.uv_override = r[3];
            } else if (A.synth_seeds) {
                unsigned seed = A.synth_seeds[s];
                if (seed == 0u) {
                    seed = 0x6d25357bu;
                }
                ws.rng.comfort = (((unsigned long long)seed) ^ 0x5DEECE66DULL) & ((1ULL << 48) - 1ULL);
                ws.rng.uv_seed = seed % 53125u;
                ws.rng.uv_override = 1;
            } else {
                ws.rng.comfort = (0x12345678ULL ^ 0x5DEECE66DULL) & ((1ULL << 48) - 1ULL);
                ws.rng.uv_seed = 3147u;
                ws.rng.uv_override = 0;
            }
        }
        __syncwarp();
        go = synth_begin(ws, reinterpret_cast<const float*>(gc + OVERLAP_WORD), T, 0, 0.0f, lane);
    }
    if (threadIdx.x == 0) {
        bs->n_interp[0] = 0;
    }
    __syncthreads();
    publish_components(bs, 0, ws, go, warp, lane);
    __syncthreads();
    StageTimer tm;
    voiced_bank_block(wsa, bs, 0, bt, T, tm, warp, lane);
    if (live) {
        if (go) {
            synth_finish_a(ws, gc, nullptr, T, bt, lane);
            const WolaTail tail = synth_finish_b(ws, gp, bt, lane);
            synth_finish_c(ws, gc, nullptr, tail, bt, lane);
        }
        __syncwarp();
        store_pcm(A, ws, (size_t)s, lane);
        for (int i = lane; i < HEAD_WORDS; i += 32) {
            gc[i] = ref_nan_parms_word(i, c[i]);
        }
        for (int j = lane; j < ENH_WORDS; j += 32) {
            gp[enh_word(j)] = ref_nan_parms_word(enh_word(j), e[j]);
        }
        if (lane == 0) {
            gc[SEED_WORD] = c[HEAD_WORDS];
            if (A.synth_rng) {
                uint32_t* r = A.synth_rng + 4 * (size_t)s;
                r[0] = (uint32_t)(ws.rng.comfort & 0xffffffffULL);
                r[1] = (uint32_t)(ws.rng.comfort >> 32);
                r[2] = ws.rng.uv_seed;
                r[3] = ws.rng.uv_override;
            }
        }
    }
}

// Single stages of the path on caller-held parameter sets (batched mbe_decode<Codec>Parms, mbe_spectralAmpEnhance,
// mbe_applyAdaptiveSmoothing; mbelib.h:301,385,461,623,725): the same device functions the stream kernel fuses, one warp
// per element, so that rows P1-P5 of SURVEY 8(a) can be checked on their own.  No block barriers.
// STAGE_TONE: mbe_synthesizeTonef (tone_id == nullptr: indices parsed from the 49 parameter bits) / mbe_synthesizeTonefdstar
// (tone_id[i] = ID1) into pcmf, tone phases of cur updated; STAGE_COMFORT: mbe_synthesizeComfortNoisef with the caller's RNG
// words in `rng` (in/out) instead of cur.
enum { STAGE_PARMS_IMBE = 0, STAGE_PARMS_A2400 = 1, STAGE_PARMS_A2450 = 2, STAGE_ENHANCE = 3, STAGE_SMOOTH = 4, STAGE_TONE = 5,
       STAGE_COMFORT = 6 };
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32, MIN_BLOCKS_PER_SM)
mbe_stage_kernel(int op, int n, const uint8_t* __restrict__ bits, uint32_t* cur, uint32_t* prev, int32_t* status, float* rm0,
                 float* pcmf, const int32_t* tone_id, uint32_t* rng, const DevTables* T) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    WarpWS* wsa = reinterpret_cast<WarpWS*>(smem_raw + sizeof(BlockTables));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int s = blockIdx.x * WARPS_PER_BLOCK + warp;
    if (s >= n) {
        return;
    }
    WarpWS& ws = wsa[warp];
    if (op == STAGE_COMFORT) {
        uint32_t* r = rng + 4 * (size_t)s;
        if (lane == 0) {
            ws.rng.comfort = (unsigned long long)r[0] | ((unsigned long long)r[1] << 32);
        }
        __syncwarp();
        comfort_noise(ws, T, lane);
        for (int i = lane; i < NS; i += 32) {
            pcmf[(size_t)s * NS + i] = ref_nan(ws.out[i]);
        }
        if (lane == 0) {
            r[0] = (uint32_t)(ws.rng.comfort & 0xffffffffULL);
            r[1] = (uint32_t)(ws.rng.comfort >> 32);
        }
        return;
    }
    uint32_t* gc = cur + (size_t)s * PARMS_WORDS;
    uint32_t* gp = prev ? prev + (size_t)s * PARMS_WORDS : nullptr;
    uint32_t* c = reinterpret_cast<uint32_t*>(&ws.cur);
    uint32_t* p = reinterpret_cast<uint32_t*>(&ws.prev);
    uint32_t* e = reinterpret_cast<uint32_t*>(&ws.enh);
    for (int i = lane; i < HEAD_WORDS; i += 32) {
        c[i] = gc[i];
    }
    if (lane == 0) {
        c[HEAD_WORDS] = gc[SEED_WORD];
        ws.w0row = ws.w0row_prev = ws.w0row_enh = -1;
    }
    if (op <= STAGE_PARMS_A2450) {
        for (int j = lane; j < PREV_WORDS; j += 32) {
            p[j] = gp[prev_word(j)];
        }
    } else if (op == STAGE_SMOOTH) {
        for (int j = lane; j < ENH_WORDS; j += 32) {
            e[j] = gp[enh_word(j)];
        }
    }
    __syncwarp();
    int rc = 0;
    if (op <= STAGE_PARMS_A2450) {
        const int pbits = (op == STAGE_PARMS_IMBE) ? 88 : 49;
        const uint8_t* d = bits + (size_t)s * pbits;
        unsigned dw[3];
        bool bad = false;
#pragma unroll
        for (int w = 0; w < 3; ++w) {
            const int i = 32 * w + lane;
            unsigned b = 0;
            if (i < pbits) {
                const unsigned v = d[i];
                bad |= (v > 1u);
                b = v & 1u;
            }
            dw[w] = __ballot_sync(FULL, b);
        }
        if (__any_sync(FULL, bad)) {
            rc = -2;  // MBE_STATUS_INVALID_BITS, nothing touched
        } else if (op == STAGE_PARMS_IMBE) {
            rc = decode_imbe(dw, ws, T, lane);
        } else if (op == STAGE_PARMS_A2400) {
            rc = decode_ambe2400(dw, ws, T, lane);
        } else {
            rc = decode_ambe2450(dw, ws, T, -1, lane);  // the public wrapper passes "no error count" (ambe3600x2450.c:630-633)
        }
    } else if (op == STAGE_ENHANCE) {
        const float r = spectral_enhance(ws, T, reinterpret_cast<float*>(&ws.u), lane);
        if (rm0 && lane == 0) {
            rm0[s] = r;
        }
    } else if (op == STAGE_TONE) {
        // mbelib.c:762-856: invalid bits, unknown tone ids and (D-STAR) anything but the single tones give silence
        const uint8_t* d = bits + (size_t)s * 49;
        unsigned dw[3] = {0u, 0u, 0u};
        bool bad = false;
#pragma unroll
        for (int w = 0; w < 2; ++w) {
            const int i = 32 * w + lane;
            unsigned b = 0;
            if (i < 49) {
                const unsigned v = d[i];
                bad |= (v > 1u);
                b = v & 1u;
            }
            dw[w] = __ballot_sync(FULL, b);
        }
        float f1 = 0.0f, f2 = 0.0f;
        int amp = 103;
        bool ok;
        if (tone_id) {
            const int id = tone_id[s];
            ok = (id >= 5 && id <= 122) && tone_freqs(id, &f1, &f2);
        } else {
            unsigned u0 = 0, u1 = 0, u3 = 0;
            for (int i = 0; i < 12; ++i) {
                u0 = (u0 << 1) | getbit(dw, i);
            }
            for (int i = 12; i < 24; ++i) {
                u1 = (u1 << 1) | getbit(dw, i);
            }
            for (int i = 35; i < 49; ++i) {
                u3 = (u3 << 1) | getbit(dw, i);
            }
            amp = (int)(((u0 & 0x3fu) << 1) + ((u3 >> 4) & 1u));
            ok = !__any_sync(FULL, bad) && tone_freqs((int)((u1 & 0xfffu) >> 4), &f1, &f2);
        }
        render_tone(ws, ok ? f1 : 0.0f, f2, amp, lane);
        for (int i = lane; i < NS; i += 32) {
            pcmf[(size_t)s * NS + i] = ref_nan(ws.out[i]);
        }
    } else {
        adaptive_smoothing(ws.cur, ws.enh, 0, 0.0f, lane);
    }
    __syncwarp();
    for (int i = lane; i < HEAD_WORDS; i += 32) {
        gc[i] = ref_nan_parms_word(i, c[i]);
    }
    if (op <= STAGE_PARMS_A2450) {  // the decoders extend / touch prev_mp's magnitudes (SURVEY 8(a) trap T3)
        for (int j = lane; j < PREV_WORDS - 1; j += 32) {
            gp[prev_word(j)] = ref_nan_parms_word(prev_word(j), p[j]);
        }
    }
    if (status && lane == 0) {
        status[s] = rc;
    }
}

// The channel front-end one step at a time on caller-held frames (batched mbe_ecc<Codec>C0, mbe_demodulate<Codec>Data,
// mbe_ecc<Codec>Data, mbe_convertImbe7100to7200): step 0 = C0 ECC in place, 1 = de-scramble in place, 2 = data ECC ->
// parameter bits, 3 = IMBE 7100 -> 7200 bit layout in place.  status = the reference's return value.  One warp per frame.
template <int CODEC>
__global__ void __launch_bounds__(256) mbe_front_step_kernel(int step, int n, uint8_t* fr, uint8_t* d, int32_t* status,
                                                             const DevTables* T) {
    __shared__ unsigned rows_s[8][8];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int i = blockIdx.x * 8 + warp;
    if (i >= n) {
        return;
    }
    constexpr int fbits = (CODEC == MBE_B200_IMBE7200X4400) ? 184 : (CODEC == MBE_B200_IMBE7100X4400 ? 168 : 96);
    constexpr int pbits = (CODEC <= MBE_B200_IMBE7100X4400) ? 88 : 49;
    const SoftScratch S = {nullptr, nullptr, nullptr};
    unsigned dw[3] = {0u, 0u, 0u};
    int rc = 0;
    if (step == 3) {
        uint8_t* dd = d + (size_t)i * 88;
        unsigned pre[3];
        bool bad = false;
#pragma unroll
        for (int w = 0; w < 3; ++w) {
            const int k = 32 * w + lane;
            unsigned b = 0;
            if (k < 88) {
                const unsigned v = dd[k];
                bad |= (v > 1u);
                b = v & 1u;
            }
            pre[w] = __ballot_sync(FULL, b);
        }
        if (__any_sync(FULL, bad)) {
            rc = -2;
        } else {
            fe_convert7100(pre, dw, T, lane);
#pragma unroll
            for (int w = 0; w < 3; ++w) {
                const int k = 32 * w + lane;
                if (k < 88) {
                    dd[k] = (uint8_t)((dw[w] >> lane) & 1u);
                }
            }
        }
    } else {
        uint8_t* f = fr + (size_t)i * fbits;
        unsigned row[8];
        if (fe_read(CODEC, 0, 0, f, row, nullptr, T, lane)) {
            rc = -2;  // MBE_STATUS_INVALID_BITS: nothing touched
        } else if (step == 2) {
            int c4;
            rc = fe_data(CODEC, 0, false, row, nullptr, S, rows_s[warp], T, lane, dw, &c4);
#pragma unroll
            for (int w = 0; w < 3; ++w) {
                const int k = 32 * w + lane;
                if (k < pbits) {
                    d[(size_t)i * pbits + k] = (uint8_t)((dw[w] >> lane) & 1u);
                }
            }
        } else {
            if (step == 0) {
                rc = fe_c0(CODEC, 0, row, nullptr, S, T, lane);
            } else {
                fe_demod(CODEC, row, T, lane);
            }
            constexpr int rows = (CODEC == MBE_B200_IMBE7200X4400) ? 8 : (CODEC == MBE_B200_IMBE7100X4400 ? 7 : 4);
            constexpr int cols = (CODEC == MBE_B200_IMBE7200X4400) ? 23 : 24;
#pragma unroll
            for (int r = 0; r < rows; ++r) {
                if (lane < cols) {
                    f[r * cols + lane] = (uint8_t)((row[r] >> lane) & 1u);
                }
            }
        }
    }
    if (lane == 0) {
        status[i] = rc;
    }
}

// stateless ECC-only kernel: one warp per frame (batched mbe_decode<Codec>[Soft]Frame)
template <int CODEC, int SOFT>
__global__ void __launch_bounds__(256) mbe_decode_kernel(int n, const uint8_t* __restrict__ frames,
                                                         uint8_t* __restrict__ bits, mbe_b200_result* __restrict__ results,
                                                         const DevTables* T) {
    __shared__ unsigned char rel[8][8 * 24];
    __shared__ __align__(16) unsigned short cp[SOFT ? 8 : 1][SOFT ? 2048 : 2];
    __shared__ unsigned ka[SOFT ? 8 : 1][64];
    __shared__ unsigned short qa[SOFT ? 8 : 1][64];
    __shared__ unsigned rows[8][8];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int i = blockIdx.x * 8 + warp;
    if (i >= n) {
        return;
    }
    constexpr int fbits = (CODEC == MBE_B200_IMBE7200X4400) ? 184 : (CODEC == MBE_B200_IMBE7100X4400 ? 168 : 96);
    constexpr int pbits = (CODEC <= MBE_B200_IMBE7100X4400) ? 88 : 49;
    unsigned dw[3];
    const SoftScratch S = {cp[SOFT ? warp : 0], ka[SOFT ? warp : 0], qa[SOFT ? warp : 0]};
    FrontResult R = front_end(CODEC, SOFT, 0, frames + (size_t)i * fbits * (SOFT ? 2 : 1), dw, rel[warp], S, rows[warp], T,
                              lane);
    if (bits && R.status >= 0) {
#pragma unroll
        for (int w = 0; w < 3; ++w) {
            const int b = 32 * w + lane;
            if (b < pbits) {
                bits[(size_t)i * pbits + b] = (uint8_t)((dw[w] >> lane) & 1u);
            }
        }
    }
    if (results && lane == 0) {
        mbe_b200_result r;
        r.status = R.status;
        r.c0_errors = R.c0;
        r.protected_errors = R.prot;
        r.c4_errors = R.c4;
        r.total_errors = R.status >= 0 ? R.c0 + R.prot : 0;
        r.flags = R.flags;
        results[i] = r;
    }
}

// batched block decoders: one warp per code word (mbe_golay2312[Soft], mbe_hamming1511[Soft],
// mbe_7100x4400hamming1511[Soft]; src/ecc/ecc.c:259-357,366-469).  CODE: 0 Golay(23,12), 1 Hamming(15,11), 2 Hamming(15,11)
// in the IMBE 7100 layout.  in: [n][len] bits or [n][len] mbe_soft_bit pairs, bit i of the word at index i; out: [n][len].
template <int CODE, int SOFT>
__global__ void __launch_bounds__(256) mbe_ecc_block_kernel(int n, const uint8_t* __restrict__ in, uint8_t* __restrict__ out,
                                                            int32_t* __restrict__ status, const DevTables* T) {
    __shared__ unsigned char rel[8][24];
    __shared__ __align__(16) unsigned short cp[SOFT ? 8 : 1][SOFT ? 2048 : 2];
    __shared__ unsigned ka[SOFT ? 8 : 1][64];
    __shared__ unsigned short qa[SOFT ? 8 : 1][64];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int i = blockIdx.x * 8 + warp;
    if (i >= n) {
        return;
    }
    constexpr int len = (CODE == 0) ? 23 : 15;
    unsigned v = 0;
    if (lane < len) {
        if (SOFT) {
            v = in[((size_t)i * len + lane) * 2];
            rel[warp][lane] = in[((size_t)i * len + lane) * 2 + 1];
        } else {
            v = in[(size_t)i * len + lane];
        }
    }
    const bool bad = __any_sync(FULL, v > 1u);
    const unsigned w = __ballot_sync(FULL, (v & 1u) != 0u);
    __syncwarp();
    if (bad) {
        if (lane == 0) {
            status[i] = -2;  // MBE_STATUS_INVALID_BITS: output untouched, like the reference
        }
        return;
    }
    const SoftScratch S = {cp[SOFT ? warp : 0], ka[SOFT ? warp : 0], qa[SOFT ? warp : 0]};
    int errs = 0;
    unsigned r;
    if (CODE == 0) {
        r = golay_row(w, rel[warp], SOFT, S, T, lane, &errs);
    } else {
        r = hamming_row<CODE == 2 ? 1 : 0>(w, rel[warp], SOFT, S, T, lane, &errs);
    }
    if (lane < len) {
        out[(size_t)i * len + lane] = (uint8_t)((r >> lane) & 1u);
    }
    if (lane == 0) {
        status[i] = errs;
    }
}

typedef void (*ecc_block_kernel_fn)(int, const uint8_t*, uint8_t*, int32_t*, const DevTables*);
static ecc_block_kernel_fn pick_ecc_block_kernel(int code, int soft) {
    switch (code * 2 + (soft ? 1 : 0)) {
        case 0: return mbe_ecc_block_kernel<0, 0>;
        case 1: return mbe_ecc_block_kernel<0, 1>;
        case 2: return mbe_ecc_block_kernel<1, 0>;
        case 3: return mbe_ecc_block_kernel<1, 1>;
        case 4: return mbe_ecc_block_kernel<2, 0>;
        default: return mbe_ecc_block_kernel<2, 1>;
    }
}

__global__ void mbe_floattoshort_kernel(size_t n, const float* __restrict__ in, int16_t* __restrict__ out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        out[i] = float_to_short(in[i]);
    }
}

// per stream: mbe_setThreadRngSeed(seed) + mbe_initMbeParms (mbelib.c:173-181,367-410)
// (slots != nullptr: element i is stream slot slots[i] - an indexed call, validated on the host - instead of first + i)
struct SlotList {
    const int32_t* slots;
    int first_stream, slot_base, io_base;
};
__global__ void mbe_init_streams_kernel(uint32_t* state, SlotList sl, int count, const uint32_t* seeds, float w0, int L) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= count) {
        return;
    }
    uint32_t* gs = state + (size_t)slot_of(sl, warp) * STATE_WORDS;
    Parms* p = reinterpret_cast<Parms*>(gs);
    for (int k = 0; k < 3; ++k) {
        fill_default(p + k, w0, L, 12, 0.0875f, lane);
    }
    if (lane == 0) {
        unsigned long long comfort;
        unsigned uvs, ovr;
        if (seeds) {
            unsigned seed = seeds[warp];
            if (seed == 0u) {
                seed = 0x6d25357bu;
            }
            comfort = (((unsigned long long)seed) ^ 0x5DEECE66DULL) & ((1ULL << 48) - 1ULL);
            uvs = seed % 53125u;
            ovr = 1;
        } else {
            comfort = (0x12345678ULL ^ 0x5DEECE66DULL) & ((1ULL << 48) - 1ULL);
            uvs = 3147u;
            ovr = 0;
        }
        gs[3 * PARMS_WORDS] = (uint32_t)(comfort & 0xffffffffULL);
        gs[3 * PARMS_WORDS + 1] = (uint32_t)(comfort >> 32);
        gs[3 * PARMS_WORDS + 2] = uvs;
        gs[3 * PARMS_WORDS + 3] = ovr;
    }
}

// gather/scatter between the interleaved HBM state pool and dense [count][3][651] / [count][4] buffers
__global__ void mbe_state_xfer_kernel(uint32_t* state, SlotList sl, int count, uint32_t* dense, int words, int offset,
                                      int to_dense) {
    const size_t total = (size_t)count * words;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t s = i / words, w = i % words;
        uint32_t* g = state + (size_t)slot_of(sl, (int)s) * STATE_WORDS + offset + w;
        if (to_dense) {
            // exported mbe_parms images carry the reference's NaN pattern (the RNG words are integers: untouched)
            dense[i] = (words == 3 * PARMS_WORDS) ? ref_nan_parms_word((int)(w % PARMS_WORDS), *g) : *g;
        } else {
            *g = dense[i];
        }
    }
}

// single-frame call (mbe_b200_single_frame): one stream's {cur, prev, enh} triplet + RNG words between a dense blob and its slot
__global__ void mbe_single_io_kernel(uint32_t* state, int stream, uint32_t* blob, int to_blob) {
    uint32_t* g = state + (size_t)stream * STATE_WORDS;
    constexpr int N = 3 * PARMS_WORDS + RNG_WORDS;   // the slot's first words are exactly these
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
        if (to_blob) {
            blob[i] = (i < 3 * PARMS_WORDS) ? ref_nan_parms_word(i % PARMS_WORDS, g[i]) : g[i];
        } else {
            g[i] = blob[i];
        }
    }
}

// indexed calls: every element whose slot is in range leaves its tag on the slot; the largest tag - the element of the call
// that lists the slot first - is the one the frame kernels accept (one launch over the whole list, so a repeated slot is
// caught wherever the host pipeline cuts the list into chunks)
__global__ void mbe_claim_kernel(const int32_t* slots, int n, int max_streams, unsigned long long* claim, unsigned epoch) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int slot = slots[i];
        if ((unsigned)slot < (unsigned)max_streams) {
            atomicMax(&claim[slot], claim_tag(epoch, i));
        }
    }
}

}  // namespace mbe

// =====================================================================================================
// Host side
// =====================================================================================================
using namespace mbe;

// the host-pointer entry points cut a batch into up to MAX_CHUNKS stream ranges and pipeline them
constexpr int MAX_CHUNKS = 64;
constexpr int MAX_KSTREAMS = 4;
constexpr int KT_MAX = 8192;                        // launches a timing session can hold
constexpr int MAX_AUX = 4;                          // internal streams of a two-kernel-path launch on a caller's stream
constexpr int DESC_SLOTS = MAX_KSTREAMS + MAX_AUX;  // descriptor buffers: one per pipeline compute stream, one per internal stream

struct mbe_b200_ctx {
    int device;
    int max_streams;
    int pending;           // an mbe_b200_submit_frames batch has not been waited for yet
    int chan_bits[4];      // transmitted bits per bit-packed frame (channel map; default = rows * cols)
    int normalized_float;  // float PCM outputs scaled by 7/32768 (mbelib.h:16-20) instead of the historical scale
    uint32_t* d_state;
    DevTables* d_tab;
    cudaStream_t stream;
    // host-pointer pipeline: copy-in stream, compute streams taken in rotation, copy-out stream, chunk events
    cudaStream_t s_in, s_k[MAX_KSTREAMS], s_out;
    cudaEvent_t ev_in[MAX_CHUNKS], ev_k[MAX_CHUNKS], ev_start;
    // staging for the host-pointer entry points (grown on demand)
    void* d_in;
    size_t d_in_cap;
    void* d_out[4];
    size_t d_out_cap[4];
    long long launches;
    unsigned long long* d_dbg;  // 16 stage counters (MBE_STAGE_TIMING builds)
    float imbe_default_w0;
    int imbe_default_L;
    // two-kernel path (mbe_split.cuh): descriptor buffers, one per pipeline compute stream + one shared by every other
    // stream; a buffer is reused only after the synthesis kernel that read it has finished (ev_desc)
    int split;
    void* d_desc[DESC_SLOTS];
    size_t d_desc_cap[DESC_SLOTS];
    cudaEvent_t ev_desc[DESC_SLOTS];
    // launches on any other stream fork their stream ranges over these, so that the parameter kernel of one range runs
    // while the bank / unvoiced kernels of the previous ones do (slots MAX_KSTREAMS.. of d_desc)
    cudaStream_t s_aux[MAX_AUX];
    cudaEvent_t ev_fork, ev_join[MAX_AUX];
    // per-kernel device time (mbe_b200_set_kernel_timing): an event pair around every launch of the frame kernels
    // mbe_b200_single_frame: one pinned host blob and its device twin (state + RNG + frame in, PCM + result + bits out)
    unsigned char* h_one;
    unsigned char* d_one;
    int force_fused;       // the single-frame call runs the fused kernel (one launch instead of three + fork / join)
    int kt_on, kt_n;
    cudaEvent_t* kt_ev;               // [2 * KT_MAX]
    unsigned char* kt_kind;           // [KT_MAX]: 0 parameter (or fused) kernel, 1 bank kernel, 2 unvoiced kernel
    unsigned long long* d_cnt;        // [6] device counters of the bank kernel ([0..3]) and the unvoiced kernel ([4..5])
    // noise spectrum table of the unvoiced kernel (mbe_noise_table_kernel): built on the first multi-kernel launch
    float* d_noise_tab;
    cudaEvent_t ev_noise_tab;         // the build is done (launches on the pipeline's compute streams wait for it)
    // indexed calls: the claim tag of every slot (mbe_claim_kernel), the epoch of the latest call, and the device copy of a
    // host slot list (reused like d_in: host-pointer calls are synchronous or pending until mbe_b200_wait)
    unsigned long long* d_claim;      // [max_streams]
    unsigned claim_epoch;
    int32_t* d_slots;
    size_t d_slots_cap;
    char err[256];
};

static char g_create_err[256] = "";

static int fail(mbe_b200_ctx* ctx, int code, const char* what, cudaError_t ce) {
    char* dst = ctx ? ctx->err : g_create_err;
    if (ce != cudaSuccess) {
        snprintf(dst, 256, "%s: %s", what, cudaGetErrorString(ce));
    } else {
        snprintf(dst, 256, "%s", what);
    }
    return code;
}

#define CU(call)                                                 \
    do {                                                         \
        cudaError_t _e = (call);                                 \
        if (_e != cudaSuccess) {                                 \
            return fail(ctx, MBE_B200_E_CUDA, #call, _e);        \
        }                                                        \
    } while (0)

static void build_tables(DevTables* t) {
    memset(t, 0, sizeof(*t));
    // DCT cosine tables.  The reference's Release build (gcc -O3) constant-folds the 6x6 gain table, so
    // those entries are correctly rounded cosines ((float)cos((double)x) reproduces all 36); the 8x8 and
    // per-block tables come from glibc's cosf at run time (imbe7200x4400.c:97-111, ambe3600x2450.c:60-74).
    for (int m = 1; m <= 6; ++m) {
        for (int i = 1; i <= 6; ++i) {
            float arg = (M_PI * (float)(m - 1) * ((float)i - 0.5f)) / 6.0f;
            t->ri6[(m - 1) * 6 + (i - 1)] = (float)cos((double)arg);
        }
    }
    for (int m = 1; m <= 8; ++m) {
        for (int i = 1; i <= 8; ++i) {
            t->ri8[(m - 1) * 8 + (i - 1)] = cosf((M_PI * (float)(m - 1) * ((float)i - 0.5f)) / 8.0f);
        }
    }
    int off = 0;
    for (int ji = 1; ji <= 17; ++ji) {
        t->blk_off[ji] = off;
        for (int j = 1; j <= ji; ++j) {
            for (int k = 1; k <= ji; ++k) {
                t->blk[off + (j - 1) * ji + (k - 1)] = cosf((M_PI * (float)(k - 1) * ((float)j - 0.5f)) / (float)ji);
            }
        }
        off += ji * ji;
    }
    // FFTPACK twiddles, N = 256, factors 4x4x4x4 (pffft.c:1231-1262)
    {
        const int n = 256;
        float argh = (2 * M_PI) / n;
        int is = 0, l1 = 1;
        for (int pass = 1; pass <= 3; ++pass) {
            int l2 = l1 * 4, ido = n / l2, ld = 0;
            for (int j = 1; j <= 3; ++j) {
                int i = is, fi = 0;
                ld += l1;
                float argld = ld * argh;
                for (int ii = 3; ii <= ido; ii += 2) {
                    i += 2;
                    fi += 1;
                    // C semantics: double cos/sin of the float product (C++ would pick the float overload)
                    t->tw[i - 2] = (float)cos((double)(fi * argld));
                    t->tw[i - 1] = (float)sin((double)(fi * argld));
                }
                is += ido;
            }
            l1 = l2;
        }
    }
    // b0 -> (w0, L, K)  (imbe7200x4400.c:117-154, imbe7100x4400.c:392-402)
    for (int b0 = 0; b0 < 256; ++b0) {
        float w0 = ((float)(4 * M_PI) / (float)((float)b0 + 39.5));
        int L = (int)(0.9254 * (int)((M_PI / w0) + 0.25));
        int K = (L < 37) ? (int)((float)(L + 2) / (float)3) : 12;
        t->imbe_w0[b0] = w0;
        t->imbe_K[b0] = (unsigned char)K;
        t->imbe_Kv[b0] = (unsigned char)K;
        t->imbe_L[b0] = (b0 <= 207 && L >= 9 && L <= 56) ? (unsigned char)L : 0;
    }
    for (int b0 = 0; b0 < 120; ++b0) {
        t->a2450_w0[b0] = hosttab::t_a2450_f0[b0] * (float)2 * M_PI;
    }
    t->a2450_f0_silence = (float)M_PI / 32.0f;
    t->a2450_w0_silence = t->a2450_f0_silence * (float)(2.0 * M_PI);
    for (int b0 = 0; b0 < 126; ++b0) {
        float f0 = exp2f(-4.311767578125f - (2.1336e-2f * ((float)b0 + 0.5f)));
        t->a2400_f0[b0] = f0;
        t->a2400_w0[b0] = f0 * (float)2 * M_PI;
    }
    t->a2400_w0_silence = ((float)2 * M_PI) / (float)32;
    t->imbe_default_w0 = (float)((4.0 * M_PI) / (134.0 + 39.5));
    t->imbe_default_L = (int)(0.9254 * (int)((M_PI / t->imbe_default_w0) + 0.25));
    t->ambe_default_w0 = (float)((M_PI / 32.0) * (2.0 * M_PI));
    for (int L = 1; L <= 56; ++L) {
        t->log2_int[L] = log2f((float)L);
    }
    t->ambe_rconst = ((float)1 / ((float)2 * M_SQRT2));
    // LCG jump-ahead coefficients
    {
        unsigned a = 1, c = 0;
        for (int k = 0; k < 116; ++k) {
            t->pnA[k] = (unsigned short)a;
            t->pnC[k] = (unsigned short)c;
            c = (173u * c + 13849u) & 0xffffu;
            a = (173u * a) & 0xffffu;
        }
    }
    {
        unsigned long long a = 1, c = 0;
        for (int k = 0; k <= 160; ++k) {
            t->uvA[k] = (unsigned)a;
            t->uvC[k] = (unsigned)c;
            c = (171ull * c + 11213ull) % 53125ull;
            a = (171ull * a) % 53125ull;
        }
    }
    {
        unsigned long long a = 1, c = 0;
        for (int k = 0; k < NOISE_ROWS; ++k) {
            if (k >= NOISE_ROWS - 96) {
                t->uvBA[k - (NOISE_ROWS - 96)] = (unsigned)a;
                t->uvBC[k - (NOISE_ROWS - 96)] = (unsigned)c;
            }
            c = (171ull * c + 11213ull) % 53125ull;
            a = (171ull * a) % 53125ull;
        }
    }
    {
        const unsigned long long M = (1ULL << 48) - 1ULL, MUL = 0x5DEECE66DULL, ADD = 0xBULL;
        unsigned long long a = 1, c = 0;
        for (int k = 0; k <= 160; ++k) {
            t->cnA[k] = a;
            t->cnC[k] = c;
            c = (MUL * c + ADD) & M;
            a = (MUL * a) & M;
        }
    }
    // Golay(23,12)
    for (int v = 0; v < 64; ++v) {
        unsigned hi = 0, lo = 0;
        for (int i = 0; i < 6; ++i) {
            if (v & (0x20 >> i)) {
                hi ^= hosttab::t_golay_gen[i];      // data bits 11..6
                lo ^= hosttab::t_golay_gen[6 + i];  // data bits 5..0
            }
        }
        t->golay_par_hi[v] = (unsigned short)hi;
        t->golay_par_lo[v] = (unsigned short)lo;
    }
    for (unsigned d = 0; d < 4096; ++d) {
        t->golay_cw[d] = (d << 11) | (unsigned)(t->golay_par_hi[d >> 6] ^ t->golay_par_lo[d & 63]);
    }
    memcpy(t->golay_fix, hosttab::t_golay_fix, sizeof(t->golay_fix));
    for (int c = 0; c < 4; ++c) {
        for (int i = 0; i < 184; ++i) {
            t->chan_src[c][i] = (unsigned short)i;
        }
    }
    // Hamming(15,11), standard and IMBE-7100 layouts (ecc_const.c:17-19, ecc.c:133-136)
    {
        const unsigned short rows[2][4] = {{0x7f08, 0x78e4, 0x66d2, 0x55b1}, {0x7ac8, 0x3d64, 0x1eb2, 0x7591}};
        const int dpos[2][11] = {{2, 4, 5, 6, 8, 9, 10, 11, 12, 13, 14}, {4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14}};
        const int ppos[2][4] = {{0, 1, 3, 7}, {0, 1, 2, 3}};
        for (int v = 0; v < 2; ++v) {
            for (int i = 0; i < 4; ++i) {
                t->ham_rows[v][i] = rows[v][i];
            }
            for (int syn = 0; syn < 16; ++syn) {
                unsigned flip = 0;
                for (int b = 0; b < 15 && !flip && syn; ++b) {
                    int col = 0;
                    for (int i = 0; i < 4; ++i) {
                        col |= ((rows[v][i] >> b) & 1) << i;
                    }
                    if (col == syn) {
                        flip = 1u << b;
                    }
                }
                t->ham_flip[v][syn] = (unsigned short)flip;
            }
            for (unsigned d = 0; d < 2048; ++d) {
                unsigned cw = 0;
                for (int i = 0; i < 11; ++i) {
                    cw |= ((d >> i) & 1u) << dpos[v][i];
                }
                int found = 0;
                for (int p = 0; p < 16 && !found; ++p) {
                    unsigned c = cw;
                    for (int i = 0; i < 4; ++i) {
                        c |= (unsigned)((p >> i) & 1) << ppos[v][i];
                    }
                    int syn = 0;
                    for (int i = 0; i < 4; ++i) {
                        syn |= (__builtin_popcount(c & rows[v][i]) & 1) << i;
                    }
                    if (syn == 0) {
                        cw = c;
                        found = 1;
                    }
                }
                t->ham_cw[v][d] = (unsigned short)cw;
            }
            // parity bits of a codeword, compacted, as a linear function of the two halves of its data index
            for (unsigned d = 0; d < 64; ++d) {
                unsigned lo = 0, hi = 0;
                for (int i = 0; i < 4; ++i) {
                    lo |= ((unsigned)(t->ham_cw[v][d] >> ppos[v][i]) & 1u) << i;
                    if (d < 32) {
                        hi |= ((unsigned)(t->ham_cw[v][d << 6] >> ppos[v][i]) & 1u) << i;
                    }
                }
                t->ham_par_lo[v][d] = (unsigned char)lo;
                if (d < 32) {
                    t->ham_par_hi[v][d] = (unsigned char)hi;
                }
            }
        }
    }
    // windows (mbe_unvoiced_fft.c:159-176)
    for (int i = 0; i < 256; ++i) {
        int n = i - 128;
        t->uvwin[i] = (n >= -105 && n <= 105) ? hosttab::t_win_unvoiced[n + 105] : 0.0f;
    }
    for (int n = 0; n < 160; ++n) {
        float wp = (n <= 105) ? hosttab::t_win_unvoiced[n + 105] : 0.0f;
        int m = n - 160;
        float wc = (m >= -105) ? hosttab::t_win_unvoiced[m + 105] : 0.0f;
        t->wola_wp[n] = wp;
        t->wola_wc[n] = wc;
        float wp2 = wp * wp, wc2 = wc * wc;
        t->wola_den[n] = wp2 + wc2;
    }
    for (int i = 0; i < 321; ++i) {
        t->voiced_win[i] = hosttab::t_win_voiced[i];
    }
}

// Tuning knobs from the environment, read ONCE (the pool calls the host-pointer entry points from one thread per shard):
//   MBE_B200_PAD_SMEM  bytes of extra dynamic shared memory per block (profiling: lowers occupancy without touching code)
//   MBE_B200_CHUNKS    target number of pipeline chunks of a host-pointer call
//   MBE_B200_TAPER     smallest piece of the tapered ends, in blocks (0 = no taper)
//   MBE_B200_KSTREAMS  compute streams the chunks rotate over
struct Knobs {
    long pad_smem;
    int chunks, taper_blocks, kstreams;
    int aux_streams;  // MBE_B200_AUX: internal streams a multi-kernel launch forks its stream ranges over
    int split;        // MBE_B200_SPLIT: default kernel path of new contexts (0 fused, 1 parameter + synthesis kernels)
    long desc_mb;     // MBE_B200_DESC_MB: descriptor buffer budget per launch, MiB
    int skip_kernels; // MBE_B200_SKIP_KERNELS (timing experiments only, results are wrong): 1 parameter (after the first use of
                      // a descriptor buffer), 2 bank, 4 unvoiced kernel launches are skipped
    int noise_table;  // MBE_B200_NOISE_TABLE: 0 = the unvoiced kernel computes every noise spectrum (no 54 MB table per context)
};
static Knobs g_knobs;
static std::once_flag g_knobs_once;
static std::atomic<int> g_sm_count{148};   // SMs of the device of the most recently created context (B200: 148)
static const Knobs& knobs() {
    std::call_once(g_knobs_once, []() {
        const char* e = getenv("MBE_B200_PAD_SMEM");
        g_knobs.pad_smem = e ? atol(e) : 0;
        e = getenv("MBE_B200_CHUNKS");
        g_knobs.chunks = e ? atoi(e) : 0;
        e = getenv("MBE_B200_TAPER");
        g_knobs.taper_blocks = e ? atoi(e) : -1;
        e = getenv("MBE_B200_KSTREAMS");
        g_knobs.kstreams = e ? atoi(e) : 0;
        e = getenv("MBE_B200_AUX");
        g_knobs.aux_streams = e ? atoi(e) : 0;
        e = getenv("MBE_B200_SPLIT");
        g_knobs.split = e ? atoi(e) : MBE_SPLIT_DEFAULT;
        e = getenv("MBE_B200_SKIP_KERNELS");
        g_knobs.skip_kernels = e ? atoi(e) : 0;
        e = getenv("MBE_B200_NOISE_TABLE");
        g_knobs.noise_table = e ? atoi(e) : 1;
        e = getenv("MBE_B200_DESC_MB");
        g_knobs.desc_mb = e ? atol(e) : 2048;
        if (g_knobs.desc_mb < 1) {
            g_knobs.desc_mb = 1;
        }
    });
    return g_knobs;
}

static size_t stream_kernel_smem(void) {
    return sizeof(BlockTables) + (size_t)WARPS_PER_BLOCK * sizeof(WarpWS) + sizeof(BlockShared) + (size_t)knobs().pad_smem;
}
// the multi-kernel path's parameter kernel: block shape by input kind (StreamShape)
static bool parm_kernel_small(int soft) { return soft != 1; }
static int parm_kernel_warps(int soft) { return parm_kernel_small(soft) ? P_WARPS : WARPS_PER_BLOCK; }
static size_t parm_kernel_smem(int soft) {
    return parm_kernel_small(soft) ? sizeof(BlockTables) + (size_t)P_WARPS * WS_STRIDE_SMALL + (size_t)knobs().pad_smem
                                   : stream_kernel_smem();
}

typedef void (*StreamKernelFn)(const LaunchArgs);

// one kernel image per (codec, soft) for channel frames; parameter-bit input (mbe_process<Codec>Data) has no
// soft variant and IMBE 7100 shares the IMBE 4400 parameter layout
template <bool SPLIT, bool INDEXED>
static StreamKernelFn pick_stream_kernel_t(int codec, int soft, int mode) {
    if (mode == MODE_DATA) {
        switch (codec) {
            case MBE_B200_AMBE3600X2400: return mbe_stream_kernel<MBE_B200_AMBE3600X2400, 0, MODE_DATA, SPLIT, INDEXED>;
            case MBE_B200_AMBE3600X2450: return mbe_stream_kernel<MBE_B200_AMBE3600X2450, 0, MODE_DATA, SPLIT, INDEXED>;
            default: return mbe_stream_kernel<MBE_B200_IMBE7200X4400, 0, MODE_DATA, SPLIT, INDEXED>;
        }
    }
    if (soft == 2) {  // packed hard bits
        switch (codec) {
            case MBE_B200_IMBE7200X4400: return mbe_stream_kernel<MBE_B200_IMBE7200X4400, 2, MODE_FRAMES, SPLIT, INDEXED>;
            case MBE_B200_IMBE7100X4400: return mbe_stream_kernel<MBE_B200_IMBE7100X4400, 2, MODE_FRAMES, SPLIT, INDEXED>;
            case MBE_B200_AMBE3600X2400: return mbe_stream_kernel<MBE_B200_AMBE3600X2400, 2, MODE_FRAMES, SPLIT, INDEXED>;
            default: return mbe_stream_kernel<MBE_B200_AMBE3600X2450, 2, MODE_FRAMES, SPLIT, INDEXED>;
        }
    }
    switch (codec * 2 + (soft ? 1 : 0)) {
        case 0: return mbe_stream_kernel<MBE_B200_IMBE7200X4400, 0, MODE_FRAMES, SPLIT, INDEXED>;
        case 1: return mbe_stream_kernel<MBE_B200_IMBE7200X4400, 1, MODE_FRAMES, SPLIT, INDEXED>;
        case 2: return mbe_stream_kernel<MBE_B200_IMBE7100X4400, 0, MODE_FRAMES, SPLIT, INDEXED>;
        case 3: return mbe_stream_kernel<MBE_B200_IMBE7100X4400, 1, MODE_FRAMES, SPLIT, INDEXED>;
        case 4: return mbe_stream_kernel<MBE_B200_AMBE3600X2400, 0, MODE_FRAMES, SPLIT, INDEXED>;
        case 5: return mbe_stream_kernel<MBE_B200_AMBE3600X2400, 1, MODE_FRAMES, SPLIT, INDEXED>;
        case 6: return mbe_stream_kernel<MBE_B200_AMBE3600X2450, 0, MODE_FRAMES, SPLIT, INDEXED>;
        default: return mbe_stream_kernel<MBE_B200_AMBE3600X2450, 1, MODE_FRAMES, SPLIT, INDEXED>;
    }
}

static StreamKernelFn pick_stream_kernel(int codec, int soft, int mode, bool split = false, bool indexed = false) {
    if (indexed) {
        return split ? pick_stream_kernel_t<true, true>(codec, soft, mode) : pick_stream_kernel_t<false, true>(codec, soft, mode);
    }
    return split ? pick_stream_kernel_t<true, false>(codec, soft, mode) : pick_stream_kernel_t<false, false>(codec, soft, mode);
}

static size_t bank_kernel_smem(void) { return BANK_TAB_FLOATS * sizeof(float) + (size_t)B_WARPS * sizeof(BankWS); }
static size_t unvoiced_kernel_smem(void) { return sizeof(BlockTables) + 96 * sizeof(uint2) + (size_t)U_WARPS * sizeof(UnvWS); }
static size_t noise_table_smem(void) { return sizeof(BlockTables) + (size_t)NOISE_TAB_WARPS * sizeof(UnvWS); }

typedef void (*DecodeKernelFn)(int, const uint8_t*, uint8_t*, mbe_b200_result*, const DevTables*);
static DecodeKernelFn pick_decode_kernel(int codec, int soft) {
    switch (codec * 2 + (soft ? 1 : 0)) {
        case 0: return mbe_decode_kernel<MBE_B200_IMBE7200X4400, 0>;
        case 1: return mbe_decode_kernel<MBE_B200_IMBE7200X4400, 1>;
        case 2: return mbe_decode_kernel<MBE_B200_IMBE7100X4400, 0>;
        case 3: return mbe_decode_kernel<MBE_B200_IMBE7100X4400, 1>;
        case 4: return mbe_decode_kernel<MBE_B200_AMBE3600X2400, 0>;
        case 5: return mbe_decode_kernel<MBE_B200_AMBE3600X2400, 1>;
        case 6: return mbe_decode_kernel<MBE_B200_AMBE3600X2450, 0>;
        default: return mbe_decode_kernel<MBE_B200_AMBE3600X2450, 1>;
    }
}

extern "C" {

const char* mbe_b200_version(void) { return "mbe_b200 0.1.0 (sm_100a)"; }

const char* mbe_b200_last_error(const mbe_b200_ctx* ctx) { return ctx ? ctx->err : g_create_err; }

long long mbe_b200_launch_count(const mbe_b200_ctx* ctx) { return ctx ? ctx->launches : 0; }

int mbe_b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

// ---- pinned host memory for plain-C callers (no CUDA runtime on their side) -------------------------------------------
static int host_fail(const char* what, cudaError_t ce) {
    snprintf(g_create_err, sizeof(g_create_err), "%s: %s", what, cudaGetErrorString(ce));
    cudaGetLastError();
    return (ce == cudaErrorNoDevice || ce == cudaErrorInsufficientDriver) ? MBE_B200_E_NOGPU : MBE_B200_E_CUDA;
}

int mbe_b200_host_alloc(void** out, size_t bytes) {
    if (!out || bytes == 0) {
        return MBE_B200_E_ARG;
    }
    *out = nullptr;
    const cudaError_t ce = cudaHostAlloc(out, bytes, cudaHostAllocPortable);
    return ce == cudaSuccess ? 0 : host_fail("mbe_b200_host_alloc", ce);
}

int mbe_b200_host_free(void* p) {
    if (!p) {
        return 0;
    }
    const cudaError_t ce = cudaFreeHost(p);
    return ce == cudaSuccess ? 0 : host_fail("mbe_b200_host_free", ce);
}

int mbe_b200_host_register(void* p, size_t bytes) {
    if (!p || bytes == 0) {
        return MBE_B200_E_ARG;
    }
    const cudaError_t ce = cudaHostRegister(p, bytes, cudaHostRegisterPortable);
    return ce == cudaSuccess ? 0 : host_fail("mbe_b200_host_register", ce);
}

int mbe_b200_host_unregister(void* p) {
    if (!p) {
        return 0;
    }
    const cudaError_t ce = cudaHostUnregister(p);
    return ce == cudaSuccess ? 0 : host_fail("mbe_b200_host_unregister", ce);
}

int mbe_b200_geometry(int codec, int* frame_bits, int* param_bits) {
    if (codec < 0 || codec > 3) {
        return MBE_B200_E_ARG;
    }
    if (frame_bits) {
        *frame_bits = codec == 0 ? 184 : (codec == 1 ? 168 : 96);
    }
    if (param_bits) {
        *param_bits = codec <= 1 ? 88 : 49;
    }
    return 0;
}

int mbe_b200_create(mbe_b200_ctx** out, int device_ordinal, int max_streams) {
    mbe_b200_ctx* ctx = nullptr;
    if (!out || max_streams < 1) {
        return fail(nullptr, MBE_B200_E_ARG, "mbe_b200_create: bad argument", cudaSuccess);
    }
    *out = nullptr;
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev <= 0) {
        return fail(nullptr, MBE_B200_E_NOGPU, "mbe_b200_create: no CUDA device (this library has no CPU path)", ce);
    }
    if (device_ordinal < 0 || device_ordinal >= ndev) {
        return fail(nullptr, MBE_B200_E_ARG, "mbe_b200_create: device ordinal out of range", cudaSuccess);
    }
    ctx = (mbe_b200_ctx*)calloc(1, sizeof(*ctx));
    if (!ctx) {
        return fail(nullptr, MBE_B200_E_ARG, "mbe_b200_create: out of host memory", cudaSuccess);
    }
    ctx->device = device_ordinal;
    ctx->max_streams = max_streams;
    DevTables* ht = (DevTables*)malloc(sizeof(DevTables));
    build_tables(ht);
    for (int c = 0; c < 4; ++c) {
        int fb0 = 0, pb0 = 0;
        mbe_b200_geometry(c, &fb0, &pb0);
        ctx->chan_bits[c] = fb0;
    }
    ctx->imbe_default_w0 = ht->imbe_default_w0;
    ctx->imbe_default_L = ht->imbe_default_L;
#define CUC(call)                                                                  \
    do {                                                                           \
        cudaError_t _e = (call);                                                   \
        if (_e != cudaSuccess) {                                                   \
            fail(nullptr, MBE_B200_E_CUDA, #call, _e);                             \
            free(ht);                                                              \
            mbe_b200_destroy(ctx);                                                 \
            return MBE_B200_E_CUDA;                                                \
        }                                                                          \
    } while (0)
    CUC(cudaSetDevice(device_ordinal));
    {
        int sms = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device_ordinal) == cudaSuccess && sms > 0) {
            g_sm_count.store(sms);   // chunk sizes of the host pipeline are whole waves of this many SMs
        }
    }
    CUC(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    CUC(cudaStreamCreateWithFlags(&ctx->s_in, cudaStreamNonBlocking));
    for (int i = 0; i < MAX_KSTREAMS; ++i) {
        CUC(cudaStreamCreateWithFlags(&ctx->s_k[i], cudaStreamNonBlocking));
    }
    CUC(cudaStreamCreateWithFlags(&ctx->s_out, cudaStreamNonBlocking));
    CUC(cudaEventCreateWithFlags(&ctx->ev_start, cudaEventDisableTiming));
    for (int i = 0; i < MAX_CHUNKS; ++i) {
        CUC(cudaEventCreateWithFlags(&ctx->ev_in[i], cudaEventDisableTiming));
        CUC(cudaEventCreateWithFlags(&ctx->ev_k[i], cudaEventDisableTiming));
    }
    CUC(cudaMalloc(&ctx->d_tab, sizeof(DevTables)));
    // stream-ordered: a plain cudaMemcpy from pageable memory may return before its DMA has landed, and the context's
    // streams are non-blocking (no implicit ordering with the NULL stream) - the table kernel would race the upload and a
    // late DMA chunk would wipe the rows it wrote (seen as rare PCM mismatches with many contexts on one GPU)
    CUC(cudaMemcpyAsync(ctx->d_tab, ht, sizeof(DevTables), cudaMemcpyHostToDevice, ctx->stream));
    CUC(cudaStreamSynchronize(ctx->stream));
    mbe_costab_kernel<<<(COSW_ROWS + 63) / 64, 64, 0, ctx->stream>>>(ctx->d_tab);
    CUC(cudaGetLastError());
    CUC(cudaStreamSynchronize(ctx->stream));
    CUC(cudaMalloc(&ctx->d_state, (size_t)max_streams * STATE_WORDS * sizeof(uint32_t)));
    CUC(cudaMalloc(&ctx->d_dbg, 16 * sizeof(unsigned long long)));
    CUC(cudaMemsetAsync(ctx->d_dbg, 0, 16 * sizeof(unsigned long long), ctx->stream));
    CUC(cudaMalloc(&ctx->d_claim, (size_t)max_streams * sizeof(unsigned long long)));
    CUC(cudaMemsetAsync(ctx->d_claim, 0, (size_t)max_streams * sizeof(unsigned long long), ctx->stream));
    CUC(cudaStreamSynchronize(ctx->stream));
    for (int codec = 0; codec < 4; ++codec) {
        for (int soft = 0; soft < 3; ++soft) {
            for (int mode = 0; mode < (soft == 2 ? 1 : 2); ++mode) {
                for (int indexed = 0; indexed < 2; ++indexed) {
                    CUC(cudaFuncSetAttribute(pick_stream_kernel(codec, soft, mode, false, indexed),
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)stream_kernel_smem()));
                    CUC(cudaFuncSetAttribute(pick_stream_kernel(codec, soft, mode, true, indexed),
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)parm_kernel_smem(soft)));
                }
            }
        }
    }
    CUC(cudaFuncSetAttribute(mbe_synth_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)stream_kernel_smem()));
    CUC(cudaFuncSetAttribute(mbe_split_bank_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bank_kernel_smem()));
    CUC(cudaFuncSetAttribute(mbe_split_unvoiced_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)unvoiced_kernel_smem()));
    CUC(cudaFuncSetAttribute(mbe_noise_table_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)noise_table_smem()));
    for (int i = 0; i < DESC_SLOTS; ++i) {
        CUC(cudaEventCreateWithFlags(&ctx->ev_desc[i], cudaEventDisableTiming));
    }
    for (int i = 0; i < MAX_AUX; ++i) {
        CUC(cudaStreamCreateWithFlags(&ctx->s_aux[i], cudaStreamNonBlocking));
        CUC(cudaEventCreateWithFlags(&ctx->ev_join[i], cudaEventDisableTiming));
    }
    CUC(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
    CUC(cudaEventCreateWithFlags(&ctx->ev_noise_tab, cudaEventDisableTiming));
    ctx->split = knobs().split ? 1 : 0;
    CUC(cudaFuncSetAttribute(mbe_stage_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)stream_kernel_smem()));
#undef CUC
    free(ht);
    *out = ctx;
    int rc = mbe_b200_init_streams(ctx, 0, max_streams, nullptr);
    if (rc < 0) {
        snprintf(g_create_err, sizeof(g_create_err), "%s", ctx->err);
        mbe_b200_destroy(ctx);
        *out = nullptr;
        return rc;
    }
    return 0;
}

void mbe_b200_destroy(mbe_b200_ctx* ctx) {
    if (!ctx) {
        return;
    }
    cudaSetDevice(ctx->device);
    if (ctx->stream) {
        cudaStreamSynchronize(ctx->stream);
        cudaStreamDestroy(ctx->stream);
    }
    cudaStream_t extra[2 + MAX_KSTREAMS] = {ctx->s_in, ctx->s_out};
    for (int i = 0; i < MAX_KSTREAMS; ++i) {
        extra[2 + i] = ctx->s_k[i];
    }
    for (int i = 0; i < 2 + MAX_KSTREAMS; ++i) {
        if (extra[i]) {
            cudaStreamSynchronize(extra[i]);
            cudaStreamDestroy(extra[i]);
        }
    }
    if (ctx->ev_start) {
        cudaEventDestroy(ctx->ev_start);
    }
    for (int i = 0; i < MAX_CHUNKS; ++i) {
        if (ctx->ev_in[i]) {
            cudaEventDestroy(ctx->ev_in[i]);
        }
        if (ctx->ev_k[i]) {
            cudaEventDestroy(ctx->ev_k[i]);
        }
    }
    for (int i = 0; i < MAX_AUX; ++i) {
        if (ctx->s_aux[i]) {
            cudaStreamSynchronize(ctx->s_aux[i]);
            cudaStreamDestroy(ctx->s_aux[i]);
        }
        if (ctx->ev_join[i]) {
            cudaEventDestroy(ctx->ev_join[i]);
        }
    }
    if (ctx->ev_fork) {
        cudaEventDestroy(ctx->ev_fork);
    }
    if (ctx->ev_noise_tab) {
        cudaEventDestroy(ctx->ev_noise_tab);
    }
    cudaFree(ctx->d_noise_tab);
    for (int i = 0; i < DESC_SLOTS; ++i) {
        if (ctx->ev_desc[i]) {
            cudaEventDestroy(ctx->ev_desc[i]);
        }
        cudaFree(ctx->d_desc[i]);
    }
    if (ctx->kt_ev) {
        for (int i = 0; i < 2 * KT_MAX; ++i) {
            if (ctx->kt_ev[i]) {
                cudaEventDestroy(ctx->kt_ev[i]);
            }
        }
        free(ctx->kt_ev);
    }
    free(ctx->kt_kind);
    cudaFree(ctx->d_cnt);
    if (ctx->h_one) {
        cudaFreeHost(ctx->h_one);
    }
    cudaFree(ctx->d_one);
    cudaFree(ctx->d_state);
    cudaFree(ctx->d_claim);
    cudaFree(ctx->d_slots);
    cudaFree(ctx->d_dbg);
    cudaFree(ctx->d_tab);
    cudaFree(ctx->d_in);
    for (int i = 0; i < 4; ++i) {
        cudaFree(ctx->d_out[i]);
    }
    free(ctx);
}

int mbe_b200_debug_stage_cycles(mbe_b200_ctx* ctx, unsigned long long* out16, int reset) {
    if (!ctx || !out16) {
        return MBE_B200_E_ARG;
    }
    CU(cudaSetDevice(ctx->device));
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(out16, ctx->d_dbg, 16 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    if (reset) {
        CU(cudaMemset(ctx->d_dbg, 0, 16 * sizeof(unsigned long long)));
        CU(cudaDeviceSynchronize());
    }
    return 0;
}

int mbe_b200_synchronize(mbe_b200_ctx* ctx) {
    if (!ctx) {
        return MBE_B200_E_ARG;
    }
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// one mbe_b200_submit_frames batch may be in flight per context; until mbe_b200_wait() every other call is refused,
// because it would reuse the staging buffers or the stream state the in-flight kernels and copies still work on
static int check_idle(mbe_b200_ctx* ctx, const char* what) {
    if (!ctx) {
        return MBE_B200_E_ARG;
    }
    if (ctx->pending) {
        char msg[160];
        snprintf(msg, sizeof(msg), "%s: a submission is still pending (call mbe_b200_wait first)", what);
        return fail(ctx, MBE_B200_E_ARG, msg, cudaSuccess);
    }
    return 0;
}

static int ensure(mbe_b200_ctx* ctx, void** p, size_t* cap, size_t need);

static int check_range(mbe_b200_ctx* ctx, int first, int count) {
    if (!ctx) {
        return MBE_B200_E_ARG;
    }
    if (first < 0 || count < 0 || first > ctx->max_streams - count) {
        return fail(ctx, MBE_B200_E_ARG, "stream range outside the context's pool", cudaSuccess);
    }
    return 0;
}

// slot list of an indexed state call: every slot in [0, max_streams) and none listed twice, or the whole call fails
static int check_slots(mbe_b200_ctx* ctx, const int32_t* slots, int n) {
    if (!ctx) {
        return MBE_B200_E_ARG;
    }
    if (n < 0 || (n > 0 && !slots)) {
        return fail(ctx, MBE_B200_E_ARG, "slot list: bad argument", cudaSuccess);
    }
    std::vector<unsigned char> seen(n > 0 ? (size_t)ctx->max_streams : 0, 0);
    for (int i = 0; i < n; ++i) {
        const int32_t slot = slots[i];
        if (slot < 0 || slot >= ctx->max_streams || seen[slot]) {
            return fail(ctx, MBE_B200_E_ARG, "slot list: a slot is outside the context's pool or listed twice", cudaSuccess);
        }
        seen[slot] = 1;
    }
    return 0;
}

// a host slot list into the context's device copy, ordered on `st`
static int upload_slots(mbe_b200_ctx* ctx, const int32_t* slots, int n, cudaStream_t st) {
    int rc = ensure(ctx, (void**)&ctx->d_slots, &ctx->d_slots_cap, (size_t)n * sizeof(int32_t));
    if (rc < 0) {
        return rc;
    }
    CU(cudaMemcpyAsync(ctx->d_slots, slots, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    return 0;
}

// slots == nullptr: streams first .. first + count - 1; otherwise the (validated) host slot list
static int init_streams_impl(mbe_b200_ctx* ctx, int first, int count, const uint32_t* seeds, const int32_t* slots) {
    int rc;
    if (check_idle(ctx, "init_streams") < 0) {
        return MBE_B200_E_ARG;
    }
    CU(cudaSetDevice(ctx->device));
    // seeds are staged through the context's input buffer (no cudaMalloc / cudaFree pair, nothing to leak on an error path)
    uint32_t* d_seeds = nullptr;
    if (seeds) {
        if ((rc = ensure(ctx, &ctx->d_in, &ctx->d_in_cap, (size_t)count * sizeof(uint32_t))) < 0) {
            return rc;
        }
        d_seeds = (uint32_t*)ctx->d_in;
        CU(cudaMemcpyAsync(d_seeds, seeds, (size_t)count * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    }
    if (slots && (rc = upload_slots(ctx, slots, count, ctx->stream)) < 0) {
        return rc;
    }
    const SlotList sl = {slots ? ctx->d_slots : nullptr, first, 0, 0};
    const int threads = 256, wpb = threads / 32;
    mbe_init_streams_kernel<<<(count + wpb - 1) / wpb, threads, 0, ctx->stream>>>(ctx->d_state, sl, count, d_seeds,
                                                                                    ctx->imbe_default_w0,
                                                                                    ctx->imbe_default_L);
    ctx->launches++;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int mbe_b200_init_streams(mbe_b200_ctx* ctx, int first, int count, const uint32_t* seeds) {
    const int rc = check_range(ctx, first, count);
    if (rc < 0 || count == 0) {
        return rc;
    }
    return init_streams_impl(ctx, first, count, seeds, nullptr);
}

int mbe_b200_init_streams_indexed(mbe_b200_ctx* ctx, const int32_t* slots, int n, const uint32_t* seeds) {
    const int rc = check_slots(ctx, slots, n);
    if (rc < 0 || n == 0) {
        return rc;
    }
    return init_streams_impl(ctx, 0, n, seeds, slots);
}

static int state_xfer(mbe_b200_ctx* ctx, int first, int count, void* host, int words, int offset, int to_host,
                      const int32_t* slots = nullptr) {
    int rc = slots ? check_slots(ctx, slots, count) : check_range(ctx, first, count);
    if (rc < 0 || count == 0) {
        return rc;
    }
    if (!host) {
        return fail(ctx, MBE_B200_E_ARG, "NULL host buffer", cudaSuccess);
    }
    if (check_idle(ctx, "export/import") < 0) {
        return MBE_B200_E_ARG;
    }
    CU(cudaSetDevice(ctx->device));
    const size_t bytes = (size_t)count * words * sizeof(uint32_t);
    // dense staging copy in the context's input buffer; grid sized from the words that actually move (the single-stream
    // shim moves one stream's state four times per 20 ms frame)
    if ((rc = ensure(ctx, &ctx->d_in, &ctx->d_in_cap, bytes)) < 0) {
        return rc;
    }
    uint32_t* dense = (uint32_t*)ctx->d_in;
    if (!to_host) {
        CU(cudaMemcpyAsync(dense, host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    if (slots && (rc = upload_slots(ctx, slots, count, ctx->stream)) < 0) {
        return rc;
    }
    const SlotList sl = {slots ? ctx->d_slots : nullptr, first, 0, 0};
    const size_t n_words = (size_t)count * words;
    const int blocks = (int)((n_words + 255) / 256 < 1024 ? (n_words + 255) / 256 : 1024);
    mbe_state_xfer_kernel<<<blocks, 256, 0, ctx->stream>>>(ctx->d_state, sl, count, dense, words, offset, to_host);
    ctx->launches++;
    CU(cudaGetLastError());
    if (to_host) {
        CU(cudaMemcpyAsync(host, dense, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int mbe_b200_export_state(mbe_b200_ctx* ctx, int first, int count, void* parms_triplets) {
    return state_xfer(ctx, first, count, parms_triplets, 3 * PARMS_WORDS, 0, 1);
}
int mbe_b200_import_state(mbe_b200_ctx* ctx, int first, int count, const void* parms_triplets) {
    return state_xfer(ctx, first, count, const_cast<void*>(parms_triplets), 3 * PARMS_WORDS, 0, 0);
}
int mbe_b200_export_rng(mbe_b200_ctx* ctx, int first, int count, uint32_t* rng_words4) {
    return state_xfer(ctx, first, count, rng_words4, RNG_WORDS, 3 * PARMS_WORDS, 1);
}
int mbe_b200_export_state_indexed(mbe_b200_ctx* ctx, const int32_t* slots, int n, void* parms_triplets) {
    return state_xfer(ctx, 0, n, parms_triplets, 3 * PARMS_WORDS, 0, 1, slots);
}
int mbe_b200_import_state_indexed(mbe_b200_ctx* ctx, const int32_t* slots, int n, const void* parms_triplets) {
    return state_xfer(ctx, 0, n, const_cast<void*>(parms_triplets), 3 * PARMS_WORDS, 0, 0, slots);
}
int mbe_b200_export_rng_indexed(mbe_b200_ctx* ctx, const int32_t* slots, int n, uint32_t* rng_words4) {
    return state_xfer(ctx, 0, n, rng_words4, RNG_WORDS, 3 * PARMS_WORDS, 1, slots);
}
int mbe_b200_import_rng_indexed(mbe_b200_ctx* ctx, const int32_t* slots, int n, const uint32_t* rng_words4) {
    return state_xfer(ctx, 0, n, const_cast<uint32_t*>(rng_words4), RNG_WORDS, 3 * PARMS_WORDS, 0, slots);
}
int mbe_b200_import_rng(mbe_b200_ctx* ctx, int first, int count, const uint32_t* rng_words4) {
    return state_xfer(ctx, first, count, const_cast<uint32_t*>(rng_words4), RNG_WORDS, 3 * PARMS_WORDS, 0);
}

// event pair around one kernel launch when a timing session is on (kind: 0 parameter / fused, 1 bank, 2 unvoiced)
struct KernelTimer {
    mbe_b200_ctx* ctx;
    cudaStream_t st;
    int slot;
    KernelTimer(mbe_b200_ctx* c, int kind, cudaStream_t s) : ctx(c), st(s), slot(-1) {
        if (c->kt_on && c->kt_ev && c->kt_n < KT_MAX) {
            slot = c->kt_n++;
            c->kt_kind[slot] = (unsigned char)kind;
            cudaEventRecord(c->kt_ev[2 * slot], s);
        }
    }
    ~KernelTimer() {
        if (slot >= 0) {
            cudaEventRecord(ctx->kt_ev[2 * slot + 1], st);
        }
    }
};

// streams per range of a multi-kernel launch: as many as have their descriptors in one buffer, in whole waves of the
// parameter kernel
static size_t split_cap_streams(int n_frames, int soft) {
    const size_t per_stream = (size_t)n_frames * DESC_WORDS * sizeof(uint32_t);
    size_t cap_streams = ((size_t)knobs().desc_mb << 20) / per_stream;
    const int pw = parm_kernel_warps(soft);
    const size_t gran = (size_t)g_sm_count.load() * pw * (parm_kernel_small(soft) ? P_MINB : MIN_BLOCKS_PER_SM);   // one wave
    if (cap_streams >= gran) {
        cap_streams -= cap_streams % gran;
    } else if (cap_streams < (size_t)WARPS_PER_BLOCK) {
        cap_streams = WARPS_PER_BLOCK;
    }
    return cap_streams;
}

static int launch_stream_kernel(mbe_b200_ctx* ctx, const LaunchArgs& a_in, cudaStream_t st) {
    LaunchArgs a = a_in;
    a.pcmf_scale = ctx->normalized_float ? (7.0f / 32768.0f) : 1.0f;
    a.packed_bytes = a.soft != 2                ? 0
                     : a.mode == MODE_FRAMES    ? (ctx->chan_bits[a.codec] + 7) / 8
                                                : mbe_b200_packed_param_bytes(a.codec);   // packed parameter bits
    if (a.mode == MODE_SYNTH) {
        const int blocks = (a.n_streams + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK;
        mbe_synth_kernel<<<blocks, WARPS_PER_BLOCK * 32, stream_kernel_smem(), st>>>(a);
        ctx->launches++;
        CU(cudaGetLastError());
        return 0;
    }
    if (!ctx->split || ctx->force_fused) {
        const int blocks = (a.n_streams + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK;
        {
            KernelTimer kt(ctx, 0, st);
            pick_stream_kernel(a.codec, a.soft, a.mode, false, a.slots != nullptr)<<<blocks, WARPS_PER_BLOCK * 32,
                                                                                      stream_kernel_smem(), st>>>(a);
        }
        ctx->launches++;
        CU(cudaGetLastError());
        return 0;
    }
    // multi-kernel path: parameter kernel -> descriptors -> bank kernel -> unvoiced kernel, in ranges of streams whose
    // descriptors fit a buffer.  On a pipeline compute stream the ranges run one after the other on that stream (the
    // pipeline's other streams overlap them); on any other stream they are forked over internal streams, so that the
    // kernels of consecutive ranges overlap, and joined back into the caller's stream.
    int kslot = -1;
    for (int i = 0; i < MAX_KSTREAMS; ++i) {
        if (st == ctx->s_k[i]) {
            kslot = i;
        }
    }
    const size_t per_stream = (size_t)a.n_frames * DESC_WORDS * sizeof(uint32_t);
    const size_t cap_streams = split_cap_streams(a.n_frames, a.soft);
    const int pw = parm_kernel_warps(a.soft);
    int sub = (int)(cap_streams < (size_t)a.n_streams ? cap_streams : (size_t)a.n_streams);
    const int n_sub = (a.n_streams + sub - 1) / sub;
    if (n_sub > 1) {
        // equal ranges (whole blocks of the parameter kernel) instead of full ones and a small remainder
        const int even = ((a.n_streams + n_sub - 1) / n_sub + pw - 1) / pw * pw;
        if (even < sub) {
            sub = even;
        }
    }
    int n_aux = knobs().aux_streams;
    if (n_aux < 1 || n_aux > MAX_AUX) {
        n_aux = MAX_AUX;
    }
    if (n_aux > n_sub) {
        n_aux = n_sub;
    }
    const bool fork = (kslot < 0);
    int rc;
    if (knobs().noise_table && !ctx->d_noise_tab) {
        // published to the context only once the build is enqueued: a context never holds an unfilled table
        float* tab = nullptr;
        CU(cudaMalloc(&tab, (size_t)NOISE_ROWS * NFFT * sizeof(float)));
        mbe_noise_table_kernel<<<(NOISE_ROWS + NOISE_TAB_WARPS - 1) / NOISE_TAB_WARPS, NOISE_TAB_WARPS * 32, noise_table_smem(),
                                 st>>>(ctx->d_tab, tab);
        cudaError_t e = cudaGetLastError();
        if (e == cudaSuccess) {
            e = cudaEventRecord(ctx->ev_noise_tab, st);
        }
        if (e != cudaSuccess) {
            cudaFree(tab);
            return fail(ctx, MBE_B200_E_CUDA, "noise table build", e);
        }
        ctx->d_noise_tab = tab;
    }
    if (ctx->d_noise_tab) {
        // every launch, on whatever stream, is ordered after the build (which ran on the stream of the first launch); on a
        // caller's stream before the fork, so that every internal stream inherits it
        CU(cudaStreamWaitEvent(st, ctx->ev_noise_tab, 0));
    }
    if (fork) {
        CU(cudaEventRecord(ctx->ev_fork, st));
        for (int i = 0; i < n_aux; ++i) {
            CU(cudaStreamWaitEvent(ctx->s_aux[i], ctx->ev_fork, 0));
        }
    }
    StreamKernelFn pk = pick_stream_kernel(a.codec, a.soft, a.mode, true, a.slots != nullptr);
    const int n_total = a.n_streams, first0 = a.first_stream;
    for (int i = 0, o = 0; o < n_total; o += sub, ++i) {
        const int slot = fork ? MAX_KSTREAMS + (i % n_aux) : kslot;
        cudaStream_t ss = fork ? ctx->s_aux[i % n_aux] : st;
        if ((rc = ensure(ctx, &ctx->d_desc[slot], &ctx->d_desc_cap[slot], (size_t)sub * per_stream)) < 0) {
            return rc;
        }
        CU(cudaStreamWaitEvent(ss, ctx->ev_desc[slot], 0));   // the slot's previous user is done with the buffer
        const int ns = (n_total - o < sub) ? (n_total - o) : sub;
        a.first_stream = first0 + o;
        a.io_base = a_in.io_base + o;
        a.n_streams = ns;
        a.desc = (uint32_t*)ctx->d_desc[slot];
        const int skip = knobs().skip_kernels;
        if (!(skip & 1) || ctx->launches < 64) {
            KernelTimer kt(ctx, 0, ss);
            pk<<<(ns + pw - 1) / pw, pw * 32, parm_kernel_smem(a.soft), ss>>>(a);
        }
        ctx->launches++;
        CU(cudaGetLastError());
        SynthArgs sa;
        sa.first_stream = a.first_stream;
        sa.io_base = a.io_base;
        sa.n_streams = ns;
        sa.n_frames = a.n_frames;
        sa.desc = a.desc;
        sa.pcm = a.pcm;
        sa.pcmf = a.pcmf;
        sa.pcmf_scale = a.pcmf_scale;
        sa.state = a.state;
        sa.tab = a.tab;
        sa.counters = ctx->kt_on ? ctx->d_cnt : nullptr;
        sa.slots = a.slots;
        sa.slot_base = a.slot_base;
        sa.noise_tab = ctx->d_noise_tab;
        long long bank_blocks = ((long long)ns * a.n_frames + B_WARPS - 1) / B_WARPS;   // at least one frame per warp
        const long long resident = (long long)g_sm_count.load() * B_MINB;   // grid-stride warps: one resident wave is enough
        if (bank_blocks > resident) {
            bank_blocks = resident;
        }
        if (!(skip & 2)) {
            KernelTimer kt(ctx, 1, ss);
            mbe_split_bank_kernel<<<(unsigned)bank_blocks, B_WARPS * 32, bank_kernel_smem(), ss>>>(sa);
        }
        ctx->launches++;
        CU(cudaGetLastError());
        if (!(skip & 4)) {
            KernelTimer kt(ctx, 2, ss);
            mbe_split_unvoiced_kernel<<<(ns + U_WARPS - 1) / U_WARPS, U_WARPS * 32, unvoiced_kernel_smem(), ss>>>(sa);
        }
        ctx->launches++;
        CU(cudaGetLastError());
        CU(cudaEventRecord(ctx->ev_desc[slot], ss));
    }
    if (fork) {
        for (int i = 0; i < n_aux; ++i) {
            CU(cudaEventRecord(ctx->ev_join[i], ctx->s_aux[i]));
            CU(cudaStreamWaitEvent(st, ctx->ev_join[i], 0));
        }
    }
    return 0;
}

int mbe_b200_set_kernel_path(mbe_b200_ctx* ctx, int path) {
    if (!ctx || path < 0 || path > 1) {
        return ctx ? fail(ctx, MBE_B200_E_ARG, "set_kernel_path: 0 (fused) or 1 (parameter + synthesis kernels)", cudaSuccess)
                   : MBE_B200_E_ARG;
    }
    if (check_idle(ctx, "set_kernel_path") < 0) {
        return MBE_B200_E_ARG;
    }
    ctx->split = path;
    return 0;
}

int mbe_b200_kernel_path(const mbe_b200_ctx* ctx) { return ctx ? ctx->split : MBE_B200_E_ARG; }

int mbe_b200_set_kernel_timing(mbe_b200_ctx* ctx, int enable) {
    if (!ctx) {
        return MBE_B200_E_ARG;
    }
    CU(cudaSetDevice(ctx->device));
    if (enable && !ctx->kt_ev) {
        ctx->kt_ev = (cudaEvent_t*)calloc(2 * KT_MAX, sizeof(cudaEvent_t));
        ctx->kt_kind = (unsigned char*)calloc(KT_MAX, 1);
        if (!ctx->kt_ev || !ctx->kt_kind) {
            return fail(ctx, MBE_B200_E_ARG, "set_kernel_timing: out of host memory", cudaSuccess);
        }
        for (int i = 0; i < 2 * KT_MAX; ++i) {
            CU(cudaEventCreate(&ctx->kt_ev[i]));
        }
        CU(cudaMalloc(&ctx->d_cnt, 6 * sizeof(unsigned long long)));
    }
    if (enable) {
        CU(cudaDeviceSynchronize());
        CU(cudaMemsetAsync(ctx->d_cnt, 0, 6 * sizeof(unsigned long long), ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        ctx->kt_n = 0;
    }
    ctx->kt_on = enable ? 1 : 0;
    return 0;
}

int mbe_b200_kernel_timing(mbe_b200_ctx* ctx, double ms[3], long long launches[3], unsigned long long counters[4]) {
    if (!ctx || !ms || !launches || !counters) {
        return MBE_B200_E_ARG;
    }
    for (int i = 0; i < 3; ++i) {
        ms[i] = 0.0;
        launches[i] = 0;
    }
    for (int i = 0; i < 4; ++i) {
        counters[i] = 0;
    }
    if (!ctx->kt_ev) {
        return 0;
    }
    CU(cudaSetDevice(ctx->device));
    CU(cudaDeviceSynchronize());
    for (int i = 0; i < ctx->kt_n; ++i) {
        float t = 0.0f;
        CU(cudaEventElapsedTime(&t, ctx->kt_ev[2 * i], ctx->kt_ev[2 * i + 1]));
        const int k = ctx->kt_kind[i] < 3 ? ctx->kt_kind[i] : 0;
        ms[k] += (double)t;
        launches[k]++;
    }
    CU(cudaMemcpy(counters, ctx->d_cnt, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return 0;
}

int mbe_b200_noise_table_counters(mbe_b200_ctx* ctx, unsigned long long counters[2]) {
    if (!ctx || !counters) {
        return MBE_B200_E_ARG;
    }
    counters[0] = counters[1] = 0;
    if (!ctx->d_cnt) {
        return 0;
    }
    CU(cudaSetDevice(ctx->device));
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(counters, ctx->d_cnt + 4, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return 0;
}

// input kinds of the frame entry points: 0 = one byte per hard bit, 1 = mbe_soft_bit pairs, 2 = hard bits packed
// (MBE_B200_INPUT_*).  d_slots != nullptr: an indexed launch, elements slot_base .. slot_base + n_streams - 1 of the call's
// device slot list, claimed under `epoch` (first_stream is ignored).  mode MODE_DATA: parameter bits (kind 0 one byte per
// bit, 2 packed, indexed launches only), d_results is the IN/OUT decode context and d_bits is not used.
static int frames_dev_impl(mbe_b200_ctx* ctx, int codec, int kind, int first_stream, int n_streams, int n_frames,
                           const uint8_t* d_frames, int16_t* d_pcm, float* d_pcmf, mbe_b200_result* d_results,
                           uint8_t* d_bits, void* cuda_stream, const int32_t* d_slots = nullptr, int slot_base = 0,
                           unsigned epoch = 0, int mode = MODE_FRAMES);

int mbe_b200_process_frames_dev(mbe_b200_ctx* ctx, int codec, int soft, int first_stream, int n_streams, int n_frames,
                                const uint8_t* d_frames, int16_t* d_pcm, float* d_pcmf, mbe_b200_result* d_results,
                                uint8_t* d_bits, void* cuda_stream) {
    return frames_dev_impl(ctx, codec, soft ? 1 : 0, first_stream, n_streams, n_frames, d_frames, d_pcm, d_pcmf, d_results,
                           d_bits, cuda_stream);
}

int mbe_b200_process_frames_packed_dev(mbe_b200_ctx* ctx, int codec, int first_stream, int n_streams, int n_frames,
                                       const uint8_t* d_packed, int16_t* d_pcm, float* d_pcmf, mbe_b200_result* d_results,
                                       uint8_t* d_bits, void* cuda_stream) {
    return frames_dev_impl(ctx, codec, 2, first_stream, n_streams, n_frames, d_packed, d_pcm, d_pcmf, d_results, d_bits,
                           cuda_stream);
}

int mbe_b200_set_normalized_float(mbe_b200_ctx* ctx, int enable) {
    if (!ctx) {
        return MBE_B200_E_ARG;
    }
    ctx->normalized_float = enable ? 1 : 0;
    return 0;
}

int mbe_b200_channel_frame_bytes(const mbe_b200_ctx* ctx, int codec) {
    if (!ctx || codec < 0 || codec > 3) {
        return MBE_B200_E_ARG;
    }
    return (ctx->chan_bits[codec] + 7) / 8;
}

int mbe_b200_set_channel_map(mbe_b200_ctx* ctx, int codec, const uint16_t* map, int n_bits) {
    if (!ctx) {
        return MBE_B200_E_ARG;
    }
    int fb, pb;
    if (mbe_b200_geometry(codec, &fb, &pb) != 0 || (map && (n_bits < 1 || n_bits > fb))) {
        return fail(ctx, MBE_B200_E_ARG, "set_channel_map: bad argument", cudaSuccess);
    }
    unsigned short src[184];
    for (int i = 0; i < 184; ++i) {
        src[i] = map ? 0xffffu : (unsigned short)i;
    }
    if (map) {
        for (int k = 0; k < n_bits; ++k) {
            if (map[k] >= fb || src[map[k]] != 0xffffu) {
                return fail(ctx, MBE_B200_E_ARG, "set_channel_map: position out of range or used twice", cudaSuccess);
            }
            src[map[k]] = (unsigned short)k;
        }
    } else {
        n_bits = fb;
    }
    if (check_idle(ctx, "set_channel_map") < 0) {
        return MBE_B200_E_ARG;
    }
    CU(cudaSetDevice(ctx->device));
    CU(cudaDeviceSynchronize());  // configuration call: no launch of this device may still be reading the old map
    CU(cudaMemcpyAsync(&ctx->d_tab->chan_src[codec][0], src, sizeof(src), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));   // (the pipeline streams are non-blocking: the upload must have landed)
    ctx->chan_bits[codec] = n_bits;
    return 0;
}

int mbe_b200_packed_frame_bytes(int codec) {
    int fb, pb;
    if (mbe_b200_geometry(codec, &fb, &pb) != 0) {
        return MBE_B200_E_ARG;
    }
    return (fb + 7) / 8;
}

int mbe_b200_packed_param_bytes(int codec) {
    int fb, pb;
    if (mbe_b200_geometry(codec, &fb, &pb) != 0) {
        return MBE_B200_E_ARG;
    }
    return (pb + 7) / 8;
}

static int frames_dev_impl(mbe_b200_ctx* ctx, int codec, int kind, int first_stream, int n_streams, int n_frames,
                           const uint8_t* d_frames, int16_t* d_pcm, float* d_pcmf, mbe_b200_result* d_results,
                           uint8_t* d_bits, void* cuda_stream, const int32_t* d_slots, int slot_base, unsigned epoch,
                           int mode) {
    const int soft = kind;
    int rc = d_slots ? (ctx ? 0 : MBE_B200_E_ARG) : check_range(ctx, first_stream, n_streams);
    if (rc < 0) {
        return rc;
    }
    if (codec < 0 || codec > 3 || n_frames < 0 || !d_frames) {
        return fail(ctx, MBE_B200_E_ARG, mode == MODE_DATA ? "process_data: bad argument" : "process_frames: bad argument",
                    cudaSuccess);
    }
    if (n_streams == 0 || n_frames == 0) {
        return 0;
    }
    CU(cudaSetDevice(ctx->device));
    LaunchArgs a;
    memset(&a, 0, sizeof(a));
    a.codec = codec;
    a.soft = soft;
    a.mode = mode;
    a.first_stream = first_stream;
    a.n_streams = n_streams;
    a.n_frames = n_frames;
    a.frames = d_frames;
    a.pcm = d_pcm;
    a.pcmf = d_pcmf;
    a.results = d_results;
    a.bits = mode == MODE_FRAMES ? d_bits : nullptr;
    a.state = ctx->d_state;
    a.tab = ctx->d_tab;
    a.dbg = ctx->d_dbg;
    a.slots = d_slots;
    a.claim = ctx->d_claim;
    a.epoch = epoch;
    a.slot_base = slot_base;
    a.max_streams = ctx->max_streams;
    return launch_stream_kernel(ctx, a, cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream);
}

int mbe_b200_process_data_dev(mbe_b200_ctx* ctx, int codec, int first_stream, int n_streams, int n_frames,
                              const uint8_t* d_bits, mbe_b200_result* d_results_inout, int16_t* d_pcm, float* d_pcmf,
                              void* cuda_stream) {
    return frames_dev_impl(ctx, codec, 0, first_stream, n_streams, n_frames, d_bits, d_pcm, d_pcmf, d_results_inout, nullptr,
                           cuda_stream, nullptr, 0, 0, MODE_DATA);
}

// ---- one stream, one frame, caller-owned state: what the single-stream shim needs, as ONE upload, three kernels, ONE
// download and ONE synchronisation (the generic calls - import_state, import_rng, process_frames, export_state, export_rng -
// are ~40 runtime calls and ten synchronisations per frame, and the CUDA driver serialises the runtime calls of a process)
constexpr size_t ONE_STATE = (size_t)(3 * PARMS_WORDS + RNG_WORDS) * sizeof(uint32_t);   // triplet + RNG words
constexpr size_t ONE_FRAME = (ONE_STATE + 15) & ~(size_t)15;    // channel frame (<= 368 bytes) or parameter bits
constexpr size_t ONE_RES = ONE_FRAME + 384;                    // mbe_b200_result in / out
constexpr size_t ONE_IN_END = ONE_RES + 32;
constexpr size_t ONE_BITS = ONE_IN_END;                        // parameter bits out (<= 88)
constexpr size_t ONE_PCM = ONE_BITS + 96;                      // int16[160]
constexpr size_t ONE_PCMF = ONE_PCM + 320;                     // float[160]
constexpr size_t ONE_BYTES = ONE_PCMF + 640;
static_assert(ONE_FRAME % 16 == 0 && ONE_RES % 8 == 0 && ONE_PCM % 16 == 0 && ONE_PCMF % 16 == 0, "blob alignment");

int mbe_b200_single_frame(mbe_b200_ctx* ctx, int codec, int kind, int stream, const void* frame, void* parms_triplet,
                          uint32_t* rng_words4, int16_t* pcm, float* pcmf, mbe_b200_result* result, uint8_t* bits) {
    int rc = check_range(ctx, stream, 1);
    if (rc < 0) {
        return rc;
    }
    if (check_idle(ctx, "single_frame") < 0) {
        return MBE_B200_E_ARG;
    }
    int fb = 0, pb = 0;
    if (mbe_b200_geometry(codec, &fb, &pb) != 0 || kind < 0 || kind > 2 || !frame || !parms_triplet || !rng_words4 || (!pcm && !pcmf)) {
        return fail(ctx, MBE_B200_E_ARG, "single_frame: bad argument", cudaSuccess);
    }
    CU(cudaSetDevice(ctx->device));
    if (!ctx->h_one) {
        CU(cudaHostAlloc((void**)&ctx->h_one, ONE_BYTES, cudaHostAllocDefault));
        CU(cudaMalloc((void**)&ctx->d_one, ONE_BYTES));
        CU(cudaMemsetAsync(ctx->d_one, 0, ONE_BYTES, ctx->stream));   // (the whole blob is copied back: no uninitialised words)
        memset(ctx->h_one, 0, ONE_BYTES);
    }
    const size_t in_bytes = kind == 2 ? (size_t)pb : (size_t)fb * (kind == 1 ? 2u : 1u);
    unsigned char* h = ctx->h_one;
    unsigned char* d = ctx->d_one;
    memcpy(h, parms_triplet, 3 * sizeof(Parms));
    memcpy(h + 3 * sizeof(Parms), rng_words4, RNG_WORDS * sizeof(uint32_t));
    memcpy(h + ONE_FRAME, frame, in_bytes);
    mbe_b200_result rin;
    memset(&rin, 0, sizeof(rin));
    if (kind == 2 && result) {
        rin = *result;
    }
    memcpy(h + ONE_RES, &rin, sizeof(rin));
    cudaStream_t st = ctx->stream;
    CU(cudaMemcpyAsync(d, h, ONE_IN_END, cudaMemcpyHostToDevice, st));
    mbe_single_io_kernel<<<1, 256, 0, st>>>(ctx->d_state, stream, (uint32_t*)d, 0);
    ctx->launches++;
    CU(cudaGetLastError());
    ctx->force_fused = 1;
    if (kind == 2) {
        rc = mbe_b200_process_data_dev(ctx, codec, stream, 1, 1, d + ONE_FRAME, (mbe_b200_result*)(d + ONE_RES),
                                       pcm ? (int16_t*)(d + ONE_PCM) : nullptr, pcmf ? (float*)(d + ONE_PCMF) : nullptr, st);
    } else {
        rc = mbe_b200_process_frames_dev(ctx, codec, kind, stream, 1, 1, d + ONE_FRAME, pcm ? (int16_t*)(d + ONE_PCM) : nullptr,
                                         pcmf ? (float*)(d + ONE_PCMF) : nullptr, (mbe_b200_result*)(d + ONE_RES),
                                         d + ONE_BITS, st);
    }
    ctx->force_fused = 0;
    if (rc < 0) {
        cudaStreamSynchronize(st);
        return rc;
    }
    mbe_single_io_kernel<<<1, 256, 0, st>>>(ctx->d_state, stream, (uint32_t*)d, 1);
    ctx->launches++;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(h, d, ONE_BYTES, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    mbe_b200_result rout;
    memcpy(&rout, h + ONE_RES, sizeof(rout));
    if (result) {
        *result = rout;
    }
    if (rout.status < 0) {
        return 0;   // the reference returns before it touches the state, the bit vector or the samples
    }
    memcpy(parms_triplet, h, 3 * sizeof(Parms));
    memcpy(rng_words4, h + 3 * sizeof(Parms), RNG_WORDS * sizeof(uint32_t));
    if (bits && kind != 2) {
        memcpy(bits, h + ONE_BITS, (size_t)pb);
    }
    if (pcm) {
        memcpy(pcm, h + ONE_PCM, NS * sizeof(int16_t));
    }
    if (pcmf) {
        memcpy(pcmf, h + ONE_PCMF, NS * sizeof(float));
    }
    return 0;
}

int mbe_b200_decode_frames_dev(mbe_b200_ctx* ctx, int codec, int soft, int n, const uint8_t* d_frames, uint8_t* d_bits,
                               mbe_b200_result* d_results, void* cuda_stream) {
    if (!ctx) {
        return MBE_B200_E_ARG;
    }
    if (codec < 0 || codec > 3 || n < 0 || !d_frames) {
        return fail(ctx, MBE_B200_E_ARG, "decode_frames: bad argument", cudaSuccess);
    }
    if (n == 0) {
        return 0;
    }
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
    pick_decode_kernel(codec, soft)<<<(n + 7) / 8, 256, 0, st>>>(n, d_frames, d_bits, d_results, ctx->d_tab);
    ctx->launches++;
    CU(cudaGetLastError());
    return 0;
}

int mbe_b200_floattoshort_dev(mbe_b200_ctx* ctx, int n_frames, const float* d_in, int16_t* d_out, void* cuda_stream) {
    if (!ctx || n_frames < 0 || !d_in || !d_out) {
        return ctx ? fail(ctx, MBE_B200_E_ARG, "floattoshort: bad argument", cudaSuccess) : MBE_B200_E_ARG;
    }
    if (n_frames == 0) {
        return 0;
    }
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
    const size_t n = (size_t)n_frames * NS;
    int blocks = (int)((n + 255) / 256);
    if (blocks > 148 * 16) {
        blocks = 148 * 16;
    }
    mbe_floattoshort_kernel<<<blocks, 256, 0, st>>>(n, d_in, d_out);
    ctx->launches++;
    CU(cudaGetLastError());
    return 0;
}

// ---- host-pointer variants: stage through device buffers owned by the context ---------------------
static int ensure(mbe_b200_ctx* ctx, void** p, size_t* cap, size_t need) {
    if (need <= *cap) {
        return 0;
    }
    if (*p) {
        CU(cudaFree(*p));
        *p = nullptr;
        *cap = 0;
    }
    CU(cudaMalloc(p, need));
    *cap = need;
    return 0;
}

// Streams per pipeline chunk: half waves of the stream kernel (1 block per SM x 148 SMs x WARPS_PER_BLOCK streams),
// about thirty-two chunks per batch on four compute streams, tapered at both ends (pipeline_schedule), so the first
// copy-in and the last copy-out are the only exposed transfers and both are small
// (profiles/experiments/r01x_pipeline_taper.txt).
constexpr int PIPELINE_CHUNKS = 32;
constexpr int PIPELINE_TAPER_BLOCKS = 18;
static int pipeline_chunk_streams(int n_streams) {
    // granularity: one block per SM (half a wave): consecutive chunks run on different compute streams and share the SMs
    const int wave = g_sm_count.load() * WARPS_PER_BLOCK;
    if (n_streams <= 4 * wave) {
        return n_streams;
    }
    int target = knobs().chunks;
    if (target < 1 || target > MAX_CHUNKS) {
        target = PIPELINE_CHUNKS;
    }
    int chunk = (n_streams + target - 1) / target;
    chunk = ((chunk + wave - 1) / wave) * wave;
    while ((n_streams + chunk - 1) / chunk > MAX_CHUNKS) {
        chunk += wave;
    }
    return chunk;
}

// The chunk sizes of one call.  Body chunks of `chunk` streams; with a taper (MBE_B200_TAPER = smallest piece in
// blocks, 0 = none) the first and the last chunk's worth of streams are cut into pieces that double towards the body /
// halve towards the end, so the copy-in in front of the first kernel and the copy-out behind the last one are small.
static int pipeline_taper_blocks() {
    const int t = knobs().taper_blocks;
    return (t < 0 || t > 148) ? PIPELINE_TAPER_BLOCKS : t;
}

static int pipeline_kstreams() {
    const int k = knobs().kstreams;
    return (k < 1 || k > MAX_KSTREAMS) ? MAX_KSTREAMS : k;
}

static int pipeline_schedule(int n_streams, int chunk, int* sizes) {
    const int min_piece = pipeline_taper_blocks() * WARPS_PER_BLOCK;
    int n = 0;
    if (min_piece == 0 || n_streams < 4 * chunk) {
        for (int s0 = 0; s0 < n_streams; s0 += chunk) {
            sizes[n++] = (n_streams - s0 < chunk) ? (n_streams - s0) : chunk;
        }
        return n;
    }
    int head[8], tail[8], nh = 0, nt = 0, used = 0;
    for (int p = min_piece; p < chunk && nh < 8; p *= 2) {  // min, 2 min, 4 min ... (< chunk) at both ends
        head[nh++] = p;
        tail[nt++] = p;
        used += 2 * p;
    }
    int body = n_streams - used;
    for (int i = 0; i < nh; ++i) {
        sizes[n++] = head[i];
    }
    while (body > 0 && n < MAX_CHUNKS - nt) {
        const int left = MAX_CHUNKS - nt - n;  // chunks still available for the body
        int take = (body < chunk) ? body : chunk;
        if (left == 1) {
            take = body;
        }
        sizes[n++] = take;
        body -= take;
    }
    for (int i = nt - 1; i >= 0; --i) {
        sizes[n++] = tail[i];
    }
    return n;
}

int mbe_b200_pipeline_plan(int n_streams, int* sizes, int cap) {
    if (n_streams < 0 || (cap > 0 && !sizes)) {
        return MBE_B200_E_ARG;
    }
    if (n_streams == 0) {
        return 0;
    }
    int tmp[MAX_CHUNKS];
    const int n = pipeline_schedule(n_streams, pipeline_chunk_streams(n_streams), tmp);
    for (int i = 0; i < n && i < cap; ++i) {
        sizes[i] = tmp[i];
    }
    return n;
}

static int frames_host_impl(mbe_b200_ctx* ctx, int codec, int kind, int first_stream, int n_streams, int n_frames,
                            const uint8_t* frames, int16_t* pcm, float* pcmf, mbe_b200_result* results, uint8_t* bits,
                            bool wait = true, const int32_t* slots = nullptr, int mode = MODE_FRAMES);

// A new claim epoch for an indexed call and the claim launch over its whole device slot list on `st`.  After 2^32 - 1
// calls the epochs start over from a cleared claim table (nothing of the device may still read it).
static int claim_slots(mbe_b200_ctx* ctx, const int32_t* d_slots, int n, cudaStream_t st, unsigned* epoch) {
    if (++ctx->claim_epoch == 0u) {
        CU(cudaDeviceSynchronize());
        CU(cudaMemsetAsync(ctx->d_claim, 0, (size_t)ctx->max_streams * sizeof(unsigned long long), st));
        ctx->claim_epoch = 1u;
    }
    *epoch = ctx->claim_epoch;
    const int threads = 256;
    const int blocks = (n + threads - 1) / threads < 4096 ? (n + threads - 1) / threads : 4096;
    mbe_claim_kernel<<<blocks, threads, 0, st>>>(d_slots, n, ctx->max_streams, ctx->d_claim, *epoch);
    ctx->launches++;
    CU(cudaGetLastError());
    return 0;
}

static int check_indexed(mbe_b200_ctx* ctx, const char* what, int codec, int input, const int32_t* slots, int n, int n_frames,
                         const uint8_t* in) {
    if (!ctx) {
        return MBE_B200_E_ARG;
    }
    if (codec < 0 || codec > 3 || input < MBE_B200_INPUT_HARD || input > MBE_B200_INPUT_PACKED || n < 0 || n_frames < 0 ||
        (n > 0 && !slots) || !in) {
        char msg[96];
        snprintf(msg, sizeof(msg), "%s: bad argument", what);
        return fail(ctx, MBE_B200_E_ARG, msg, cudaSuccess);
    }
    return 0;
}

// the indexed calls of both modes: MODE_FRAMES (channel frames, `input` MBE_B200_INPUT_*) and MODE_DATA (parameter bits,
// `input` HARD = one byte per bit or PACKED, `results` the IN/OUT decode context, no `bits` output)
static int indexed_dev_impl(mbe_b200_ctx* ctx, const char* what, int mode, int codec, int input, const int32_t* d_slots, int n,
                            int n_frames, const uint8_t* d_in, int16_t* d_pcm, float* d_pcmf, mbe_b200_result* d_results,
                            uint8_t* d_bits, void* cuda_stream) {
    int rc = check_indexed(ctx, what, codec, input, d_slots, n, n_frames, d_in);
    if (rc < 0 || n == 0 || n_frames == 0) {
        return rc;
    }
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
    unsigned epoch = 0;
    if ((rc = claim_slots(ctx, d_slots, n, st, &epoch)) < 0) {
        return rc;
    }
    return frames_dev_impl(ctx, codec, input, 0, n, n_frames, d_in, d_pcm, d_pcmf, d_results, d_bits, st, d_slots, 0, epoch,
                           mode);
}

// wait == false: the asynchronous half (submit_*), completed by mbe_b200_wait
static int indexed_host_impl(mbe_b200_ctx* ctx, const char* what, int mode, int codec, int input, const int32_t* slots, int n,
                             int n_frames, const uint8_t* in, int16_t* pcm, float* pcmf, mbe_b200_result* results,
                             uint8_t* bits, bool wait) {
    int rc = check_indexed(ctx, what, codec, input, slots, n, n_frames, in);
    if (rc < 0) {
        return rc;
    }
    if (ctx->pending) {
        char msg[128];
        snprintf(msg, sizeof(msg), "%s: a submission is still pending (call mbe_b200_wait first)", what);
        return fail(ctx, MBE_B200_E_ARG, msg, cudaSuccess);
    }
    rc = frames_host_impl(ctx, codec, input, 0, n, n_frames, in, pcm, pcmf, results, bits, wait, slots, mode);
    if (rc == 0 && !wait) {
        ctx->pending = 1;
    }
    return rc;
}

int mbe_b200_process_indexed_dev(mbe_b200_ctx* ctx, int codec, int input, const int32_t* d_slots, int n, int n_frames,
                                 const uint8_t* d_in, int16_t* d_pcm, float* d_pcmf, mbe_b200_result* d_results,
                                 uint8_t* d_bits, void* cuda_stream) {
    return indexed_dev_impl(ctx, "process_indexed_dev", MODE_FRAMES, codec, input, d_slots, n, n_frames, d_in, d_pcm, d_pcmf,
                            d_results, d_bits, cuda_stream);
}

int mbe_b200_process_indexed(mbe_b200_ctx* ctx, int codec, int input, const int32_t* slots, int n, int n_frames,
                             const uint8_t* in, int16_t* pcm, float* pcmf, mbe_b200_result* results, uint8_t* bits) {
    return indexed_host_impl(ctx, "process_indexed", MODE_FRAMES, codec, input, slots, n, n_frames, in, pcm, pcmf, results, bits,
                             true);
}

int mbe_b200_submit_indexed(mbe_b200_ctx* ctx, int codec, int input, const int32_t* slots, int n, int n_frames,
                            const uint8_t* in, int16_t* pcm, float* pcmf, mbe_b200_result* results, uint8_t* bits) {
    return indexed_host_impl(ctx, "submit_indexed", MODE_FRAMES, codec, input, slots, n, n_frames, in, pcm, pcmf, results, bits,
                             false);
}

// parameter-bit input of the indexed data calls: packed 0 = one byte per bit, 1 = eight bits per byte (anything else fails
// check_indexed)
static int data_input(int packed) { return packed == 0 ? MBE_B200_INPUT_HARD : packed == 1 ? MBE_B200_INPUT_PACKED : -1; }

int mbe_b200_process_data_indexed_dev(mbe_b200_ctx* ctx, int codec, int packed, const int32_t* d_slots, int n, int n_frames,
                                      const uint8_t* d_bits, mbe_b200_result* d_results_inout, int16_t* d_pcm, float* d_pcmf,
                                      void* cuda_stream) {
    return indexed_dev_impl(ctx, "process_data_indexed_dev", MODE_DATA, codec, data_input(packed), d_slots, n, n_frames, d_bits,
                            d_pcm, d_pcmf, d_results_inout, nullptr, cuda_stream);
}

int mbe_b200_process_data_indexed(mbe_b200_ctx* ctx, int codec, int packed, const int32_t* slots, int n, int n_frames,
                                  const uint8_t* bits, mbe_b200_result* results_inout, int16_t* pcm, float* pcmf) {
    return indexed_host_impl(ctx, "process_data_indexed", MODE_DATA, codec, data_input(packed), slots, n, n_frames, bits, pcm,
                             pcmf, results_inout, nullptr, true);
}

int mbe_b200_submit_data_indexed(mbe_b200_ctx* ctx, int codec, int packed, const int32_t* slots, int n, int n_frames,
                                 const uint8_t* bits, mbe_b200_result* results_inout, int16_t* pcm, float* pcmf) {
    return indexed_host_impl(ctx, "submit_data_indexed", MODE_DATA, codec, data_input(packed), slots, n, n_frames, bits, pcm,
                             pcmf, results_inout, nullptr, false);
}

int mbe_b200_wait(mbe_b200_ctx* ctx) {
    if (!ctx) {
        return MBE_B200_E_ARG;
    }
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->s_out));
    for (int i = 0; i < MAX_KSTREAMS; ++i) {
        CU(cudaStreamSynchronize(ctx->s_k[i]));
    }
    ctx->pending = 0;
    return 0;
}

int mbe_b200_submit_frames(mbe_b200_ctx* ctx, int codec, int soft, int first_stream, int n_streams, int n_frames,
                           const uint8_t* frames, int16_t* pcm, float* pcmf, mbe_b200_result* results, uint8_t* bits) {
    if (ctx && ctx->pending) {
        return fail(ctx, MBE_B200_E_ARG, "submit_frames: a submission is still pending (call mbe_b200_wait first)", cudaSuccess);
    }
    const int rc = frames_host_impl(ctx, codec, soft ? 1 : 0, first_stream, n_streams, n_frames, frames, pcm, pcmf, results, bits,
                                    false);
    if (rc == 0) {
        ctx->pending = 1;
    }
    return rc;
}

int mbe_b200_process_frames(mbe_b200_ctx* ctx, int codec, int soft, int first_stream, int n_streams, int n_frames,
                            const uint8_t* frames, int16_t* pcm, float* pcmf, mbe_b200_result* results, uint8_t* bits) {
    return frames_host_impl(ctx, codec, soft ? 1 : 0, first_stream, n_streams, n_frames, frames, pcm, pcmf, results, bits);
}

int mbe_b200_process_frames_packed(mbe_b200_ctx* ctx, int codec, int first_stream, int n_streams, int n_frames,
                                   const uint8_t* packed, int16_t* pcm, float* pcmf, mbe_b200_result* results,
                                   uint8_t* bits) {
    return frames_host_impl(ctx, codec, 2, first_stream, n_streams, n_frames, packed, pcm, pcmf, results, bits);
}

// The pipelined host call of both modes.  MODE_DATA (indexed parameter-bit calls): `frames` holds parameter bits (kind 0
// one byte per bit, 2 packed), `results` is IN/OUT - each chunk's decode context goes up on s_in ahead of its kernel - and
// `bits` is unused.
static int frames_host_impl(mbe_b200_ctx* ctx, int codec, int kind, int first_stream, int n_streams, int n_frames,
                            const uint8_t* frames, int16_t* pcm, float* pcmf, mbe_b200_result* results, uint8_t* bits,
                            bool wait, const int32_t* slots, int mode) {
    int rc = slots ? 0 : check_range(ctx, first_stream, n_streams);   // (indexed: checked by check_indexed)
    if (rc == 0 && ctx->pending) {
        return fail(ctx, MBE_B200_E_ARG, "process_frames: a submission is still pending (call mbe_b200_wait first)", cudaSuccess);
    }
    if (rc < 0) {
        return rc;
    }
    if (codec < 0 || codec > 3 || n_frames < 0 || !frames) {
        return fail(ctx, MBE_B200_E_ARG, "process_frames: bad argument", cudaSuccess);
    }
    const size_t nf = (size_t)n_streams * n_frames;
    if (nf == 0) {
        return 0;
    }
    CU(cudaSetDevice(ctx->device));
    int fb, pb;
    mbe_b200_geometry(codec, &fb, &pb);
    const size_t in_per_frame = (mode == MODE_DATA) ? (size_t)(kind == 2 ? (pb + 7) / 8 : pb)
                                : (kind == 2) ? (size_t)((ctx->chan_bits[codec] + 7) / 8) : (size_t)fb * (kind == 1 ? 2 : 1);
    const size_t per_frame[4] = {pcm ? NS * sizeof(int16_t) : 0, pcmf ? NS * sizeof(float) : 0,
                                 results ? sizeof(mbe_b200_result) : 0, (bits && mode == MODE_FRAMES) ? (size_t)pb : 0};
    if ((rc = ensure(ctx, &ctx->d_in, &ctx->d_in_cap, nf * in_per_frame)) < 0) {
        return rc;
    }
    for (int i = 0; i < 4; ++i) {
        if (per_frame[i] && (rc = ensure(ctx, &ctx->d_out[i], &ctx->d_out_cap[i], nf * per_frame[i])) < 0) {
            return rc;
        }
    }
    // Pipeline over stream ranges: copy-in (s_in) -> kernel (two alternating compute streams, so the tail of
    // one chunk overlaps the head of the next) -> copy-out (s_out).  Everything is ordered after what is
    // already queued on the context's own stream; the call returns when the results are in host memory.
    void* host[4] = {pcm, pcmf, results, bits};
    int chunk = pipeline_chunk_streams(n_streams);
    if (ctx->split && knobs().chunks == 0) {
        // multi-kernel path: body chunks are whole stream ranges (whole waves of the parameter kernel), not fused-kernel waves
        const long long cap = (long long)split_cap_streams(n_frames, kind);
        // (only where a chunk holds at least one full range: smaller batches keep their ~32 small chunks, whose copies
        // overlap better than whole waves would compute - 119 M against 110 M frames/s end to end on 65 536 streams)
        if (cap > 0 && chunk >= cap) {
            const long long k = (chunk + cap / 2) / cap;
            long long c2 = k * cap;
            while ((n_streams + c2 - 1) / c2 > MAX_CHUNKS) {
                c2 += cap;
            }
            chunk = (int)c2;
        }
    }
    int sizes[MAX_CHUNKS];
    const int n_chunks = pipeline_schedule(n_streams, chunk, sizes);
    const int n_k = pipeline_kstreams();
    // a failure in the middle leaves copies into the caller's buffers queued: the pipeline streams are drained before the
    // error is returned, so the caller may free its buffers right away
    auto drain = [&]() {
        cudaStreamSynchronize(ctx->s_in);
        for (int i = 0; i < MAX_KSTREAMS; ++i) {
            cudaStreamSynchronize(ctx->s_k[i]);
        }
        cudaStreamSynchronize(ctx->s_out);
    };
    auto enqueue = [&]() -> int {
        CU(cudaEventRecord(ctx->ev_start, ctx->stream));
        CU(cudaStreamWaitEvent(ctx->s_in, ctx->ev_start, 0));
        for (int i = 0; i < MAX_KSTREAMS; ++i) {
            CU(cudaStreamWaitEvent(ctx->s_k[i], ctx->ev_start, 0));
        }
        // indexed: the slot list goes up once and is claimed as a whole ahead of the first chunk's frames (every chunk's
        // kernel waits for its copy-in, which s_in orders after the claim)
        unsigned epoch = 0;
        if (slots) {
            int rs = upload_slots(ctx, slots, n_streams, ctx->s_in);
            if (rs == 0) {
                rs = claim_slots(ctx, ctx->d_slots, n_streams, ctx->s_in, &epoch);
            }
            if (rs < 0) {
                return rs;
            }
        }
        int s0 = 0;
        for (int c = 0; c < n_chunks; s0 += sizes[c], ++c) {
            const int ns = sizes[c];
            const size_t f0 = (size_t)s0 * n_frames, fn = (size_t)ns * n_frames;
            cudaStream_t sk = ctx->s_k[c % n_k];
            CU(cudaMemcpyAsync((uint8_t*)ctx->d_in + f0 * in_per_frame, frames + f0 * in_per_frame, fn * in_per_frame,
                               cudaMemcpyHostToDevice, ctx->s_in));
            if (mode == MODE_DATA && results) {
                CU(cudaMemcpyAsync((mbe_b200_result*)ctx->d_out[2] + f0, results + f0, fn * sizeof(mbe_b200_result),
                                   cudaMemcpyHostToDevice, ctx->s_in));
            }
            CU(cudaEventRecord(ctx->ev_in[c], ctx->s_in));
            CU(cudaStreamWaitEvent(sk, ctx->ev_in[c], 0));
            int16_t* const o_pcm = pcm ? (int16_t*)ctx->d_out[0] + f0 * NS : nullptr;
            float* const o_pcmf = pcmf ? (float*)ctx->d_out[1] + f0 * NS : nullptr;
            mbe_b200_result* const o_res = results ? (mbe_b200_result*)ctx->d_out[2] + f0 : nullptr;
            uint8_t* const o_bits = bits ? (uint8_t*)ctx->d_out[3] + f0 * pb : nullptr;
            const uint8_t* const i_fr = (const uint8_t*)ctx->d_in + f0 * in_per_frame;
            const int rk = frames_dev_impl(ctx, codec, kind, first_stream + s0, ns, n_frames, i_fr, o_pcm, o_pcmf, o_res, o_bits, sk,
                                           slots ? ctx->d_slots : nullptr, s0, epoch, mode);
            if (rk < 0) {
                return rk;
            }
            CU(cudaEventRecord(ctx->ev_k[c], sk));
            CU(cudaStreamWaitEvent(ctx->s_out, ctx->ev_k[c], 0));
            for (int i = 0; i < 4; ++i) {
                if (per_frame[i]) {
                    CU(cudaMemcpyAsync((uint8_t*)host[i] + f0 * per_frame[i], (uint8_t*)ctx->d_out[i] + f0 * per_frame[i],
                                       fn * per_frame[i], cudaMemcpyDeviceToHost, ctx->s_out));
                }
            }
        }
        return 0;
    };
    if ((rc = enqueue()) < 0) {
        drain();
        return rc;
    }
    if (wait) {
        CU(cudaStreamSynchronize(ctx->s_out));
        for (int i = 0; i < MAX_KSTREAMS; ++i) {
            CU(cudaStreamSynchronize(ctx->s_k[i]));
        }
    }
    return 0;
}

int mbe_b200_process_data(mbe_b200_ctx* ctx, int codec, int first_stream, int n_streams, int n_frames,
                          const uint8_t* bits, mbe_b200_result* results_inout, int16_t* pcm, float* pcmf) {
    int rc = check_range(ctx, first_stream, n_streams);
    if (rc < 0) {
        return rc;
    }
    if (codec < 0 || codec > 3 || n_frames < 0 || !bits) {
        return fail(ctx, MBE_B200_E_ARG, "process_data: bad argument", cudaSuccess);
    }
    const size_t nf = (size_t)n_streams * n_frames;
    if (nf == 0) {
        return 0;
    }
    if (check_idle(ctx, "process_data") < 0) {
        return MBE_B200_E_ARG;
    }
    CU(cudaSetDevice(ctx->device));
    int fb, pb;
    mbe_b200_geometry(codec, &fb, &pb);
    const size_t in_bytes = nf * pb;
    const size_t ob[3] = {pcm ? nf * NS * sizeof(int16_t) : 0, pcmf ? nf * NS * sizeof(float) : 0,
                          results_inout ? nf * sizeof(mbe_b200_result) : 0};
    if ((rc = ensure(ctx, &ctx->d_in, &ctx->d_in_cap, in_bytes)) < 0) {
        return rc;
    }
    for (int i = 0; i < 3; ++i) {
        if (ob[i] && (rc = ensure(ctx, &ctx->d_out[i], &ctx->d_out_cap[i], ob[i])) < 0) {
            return rc;
        }
    }
    CU(cudaMemcpyAsync(ctx->d_in, bits, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    if (results_inout) {
        CU(cudaMemcpyAsync(ctx->d_out[2], results_inout, ob[2], cudaMemcpyHostToDevice, ctx->stream));
    }
    rc = mbe_b200_process_data_dev(ctx, codec, first_stream, n_streams, n_frames, (const uint8_t*)ctx->d_in,
                                   results_inout ? (mbe_b200_result*)ctx->d_out[2] : nullptr,
                                   pcm ? (int16_t*)ctx->d_out[0] : nullptr, pcmf ? (float*)ctx->d_out[1] : nullptr,
                                   ctx->stream);
    if (rc < 0) {
        return rc;
    }
    void* host[3] = {pcm, pcmf, results_inout};
    for (int i = 0; i < 3; ++i) {
        if (ob[i]) {
            CU(cudaMemcpyAsync(host[i], ctx->d_out[i], ob[i], cudaMemcpyDeviceToHost, ctx->stream));
        }
    }
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int mbe_b200_decode_frames(mbe_b200_ctx* ctx, int codec, int soft, int n, const uint8_t* frames, uint8_t* bits,
                           mbe_b200_result* results) {
    if (!ctx) {
        return MBE_B200_E_ARG;
    }
    if (codec < 0 || codec > 3 || n < 0 || !frames) {
        return fail(ctx, MBE_B200_E_ARG, "decode_frames: bad argument", cudaSuccess);
    }
    if (n == 0) {
        return 0;
    }
    if (check_idle(ctx, "decode_frames") < 0) {
        return MBE_B200_E_ARG;
    }
    CU(cudaSetDevice(ctx->device));
    int fb, pb, rc;
    mbe_b200_geometry(codec, &fb, &pb);
    const size_t in_bytes = (size_t)n * fb * (soft ? 2 : 1);
    const size_t bb = bits ? (size_t)n * pb : 0, rb = results ? (size_t)n * sizeof(mbe_b200_result) : 0;
    if ((rc = ensure(ctx, &ctx->d_in, &ctx->d_in_cap, in_bytes)) < 0) {
        return rc;
    }
    if (bb && (rc = ensure(ctx, &ctx->d_out[3], &ctx->d_out_cap[3], bb)) < 0) {
        return rc;
    }
    if (rb && (rc = ensure(ctx, &ctx->d_out[2], &ctx->d_out_cap[2], rb)) < 0) {
        return rc;
    }
    CU(cudaMemcpyAsync(ctx->d_in, frames, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    if (bb) {
        CU(cudaMemsetAsync(ctx->d_out[3], 0, bb, ctx->stream));
    }
    rc = mbe_b200_decode_frames_dev(ctx, codec, soft, n, (const uint8_t*)ctx->d_in, bb ? (uint8_t*)ctx->d_out[3] : nullptr,
                                    rb ? (mbe_b200_result*)ctx->d_out[2] : nullptr, ctx->stream);
    if (rc < 0) {
        return rc;
    }
    if (bb) {
        CU(cudaMemcpyAsync(bits, ctx->d_out[3], bb, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (rb) {
        CU(cudaMemcpyAsync(results, ctx->d_out[2], rb, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int mbe_b200_ecc_blocks_dev(mbe_b200_ctx* ctx, int code, int soft, int n, const uint8_t* d_in, uint8_t* d_out,
                            int32_t* d_status, void* cuda_stream) {
    if (!ctx) {
        return MBE_B200_E_ARG;
    }
    if (code < 0 || code > 2 || n < 0 || !d_in || !d_out || !d_status) {
        return fail(ctx, MBE_B200_E_ARG, "ecc_blocks: bad argument", cudaSuccess);
    }
    if (n == 0) {
        return 0;
    }
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
    pick_ecc_block_kernel(code, soft)<<<(n + 7) / 8, 256, 0, st>>>(n, d_in, d_out, d_status, ctx->d_tab);
    ctx->launches++;
    CU(cudaGetLastError());
    return 0;
}

int mbe_b200_ecc_blocks(mbe_b200_ctx* ctx, int code, int soft, int n, const uint8_t* in, uint8_t* out, int32_t* status) {
    if (!ctx) {
        return MBE_B200_E_ARG;
    }
    if (code < 0 || code > 2 || n < 0 || !in || !out || !status) {
        return fail(ctx, MBE_B200_E_ARG, "ecc_blocks: bad argument", cudaSuccess);
    }
    if (n == 0) {
        return 0;
    }
    if (check_idle(ctx, "ecc_blocks") < 0) {
        return MBE_B200_E_ARG;
    }
    CU(cudaSetDevice(ctx->device));
    const size_t len = code == 0 ? 23 : 15;
    const size_t ib = (size_t)n * len * (soft ? 2 : 1), ob = (size_t)n * len, sb = (size_t)n * sizeof(int32_t);
    int rc;
    if ((rc = ensure(ctx, &ctx->d_in, &ctx->d_in_cap, ib)) < 0 || (rc = ensure(ctx, &ctx->d_out[3], &ctx->d_out_cap[3], ob)) < 0 ||
        (rc = ensure(ctx, &ctx->d_out[2], &ctx->d_out_cap[2], sb)) < 0) {
        return rc;
    }
    CU(cudaMemcpyAsync(ctx->d_in, in, ib, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(ctx->d_out[3], out, ob, cudaMemcpyHostToDevice, ctx->stream));  // words with invalid bits keep `out`
    if ((rc = mbe_b200_ecc_blocks_dev(ctx, code, soft, n, (const uint8_t*)ctx->d_in, (uint8_t*)ctx->d_out[3],
                                      (int32_t*)ctx->d_out[2], ctx->stream)) < 0) {
        return rc;
    }
    CU(cudaMemcpyAsync(out, ctx->d_out[3], ob, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpyAsync(status, ctx->d_out[2], sb, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// op: STAGE_*; bits / prev / status / rm0 as the stage needs them (host pointers)
static int stage_impl(mbe_b200_ctx* ctx, const char* what, int op, int n, const uint8_t* bits, void* cur_parms, void* prev_parms,
                      bool prev_out, int32_t* status, float* rm0) {
    if (!ctx) {
        return MBE_B200_E_ARG;
    }
    const bool need_prev = (op != STAGE_ENHANCE), need_bits = (op <= STAGE_PARMS_A2450);
    if (n < 0 || !cur_parms || (need_prev && !prev_parms) || (need_bits && !bits)) {
        return fail(ctx, MBE_B200_E_ARG, what, cudaSuccess);
    }
    if (n == 0) {
        return 0;
    }
    if (check_idle(ctx, "stage call") < 0) {
        return MBE_B200_E_ARG;
    }
    CU(cudaSetDevice(ctx->device));
    const size_t pbytes = (size_t)n * sizeof(Parms);
    const size_t bbytes = need_bits ? (size_t)n * (op == STAGE_PARMS_IMBE ? 88 : 49) : 0;
    int rc;
    if ((rc = ensure(ctx, &ctx->d_in, &ctx->d_in_cap, 2 * pbytes + bbytes)) < 0 ||
        (rc = ensure(ctx, &ctx->d_out[2], &ctx->d_out_cap[2], (size_t)n * 8)) < 0) {
        return rc;
    }
    uint8_t* base = (uint8_t*)ctx->d_in;
    CU(cudaMemcpyAsync(base, cur_parms, pbytes, cudaMemcpyHostToDevice, ctx->stream));
    if (need_prev) {
        CU(cudaMemcpyAsync(base + pbytes, prev_parms, pbytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    if (need_bits) {
        CU(cudaMemcpyAsync(base + 2 * pbytes, bits, bbytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    int32_t* d_status = (int32_t*)ctx->d_out[2];
    float* d_rm0 = (float*)ctx->d_out[2] + n;
    const int blocks = (n + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK;
    mbe_stage_kernel<<<blocks, WARPS_PER_BLOCK * 32, stream_kernel_smem(), ctx->stream>>>(
        op, n, base + 2 * pbytes, (uint32_t*)base, need_prev ? (uint32_t*)(base + pbytes) : nullptr, d_status, d_rm0, nullptr,
        nullptr, nullptr, ctx->d_tab);
    ctx->launches++;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(cur_parms, base, pbytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (prev_out) {
        CU(cudaMemcpyAsync(prev_parms, base + pbytes, pbytes, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (status) {
        CU(cudaMemcpyAsync(status, d_status, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (rm0) {
        CU(cudaMemcpyAsync(rm0, d_rm0, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int mbe_b200_decode_parms(mbe_b200_ctx* ctx, int codec, int n, const uint8_t* bits, void* cur_parms, void* prev_parms,
                          int32_t* status) {
    if (ctx && (codec < 0 || codec > 3)) {
        return fail(ctx, MBE_B200_E_ARG, "decode_parms: bad codec", cudaSuccess);
    }
    const int op = codec <= MBE_B200_IMBE7100X4400 ? STAGE_PARMS_IMBE
                                                   : (codec == MBE_B200_AMBE3600X2400 ? STAGE_PARMS_A2400 : STAGE_PARMS_A2450);
    return stage_impl(ctx, "decode_parms: bad argument", op, n, bits, cur_parms, prev_parms, true, status, nullptr);
}

int mbe_b200_spectral_amp_enhance(mbe_b200_ctx* ctx, int n, void* cur_parms, float* rm0) {
    return stage_impl(ctx, "spectral_amp_enhance: bad argument", STAGE_ENHANCE, n, nullptr, cur_parms, nullptr, false, nullptr, rm0);
}

int mbe_b200_adaptive_smoothing(mbe_b200_ctx* ctx, int n, void* cur_parms, const void* prev_parms) {
    return stage_impl(ctx, "adaptive_smoothing: bad argument", STAGE_SMOOTH, n, nullptr, cur_parms,
                      const_cast<void*>(prev_parms), false, nullptr, nullptr);
}

int mbe_b200_synthesize_tone(mbe_b200_ctx* ctx, int n, const uint8_t* bits49, const int32_t* dstar_id, void* cur_parms,
                             float* pcmf) {
    if (!ctx) {
        return MBE_B200_E_ARG;
    }
    if (n < 0 || !cur_parms || !pcmf || (!bits49 && !dstar_id)) {
        return fail(ctx, MBE_B200_E_ARG, "synthesize_tone: bad argument", cudaSuccess);
    }
    if (n == 0) {
        return 0;
    }
    if (check_idle(ctx, "synthesize_tone") < 0) {
        return MBE_B200_E_ARG;
    }
    CU(cudaSetDevice(ctx->device));
    const size_t pbytes = (size_t)n * sizeof(Parms), bbytes = (size_t)n * 49, ibytes = (size_t)n * 4, ob = (size_t)n * NS * 4;
    int rc;
    if ((rc = ensure(ctx, &ctx->d_in, &ctx->d_in_cap, pbytes + ibytes + bbytes)) < 0 ||
        (rc = ensure(ctx, &ctx->d_out[1], &ctx->d_out_cap[1], ob)) < 0) {
        return rc;
    }
    uint8_t* base = (uint8_t*)ctx->d_in;
    CU(cudaMemcpyAsync(base, cur_parms, pbytes, cudaMemcpyHostToDevice, ctx->stream));
    if (dstar_id) {
        CU(cudaMemcpyAsync(base + pbytes, dstar_id, ibytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    if (bits49) {
        CU(cudaMemcpyAsync(base + pbytes + ibytes, bits49, bbytes, cudaMemcpyHostToDevice, ctx->stream));
    } else {
        CU(cudaMemsetAsync(base + pbytes + ibytes, 0, bbytes, ctx->stream));
    }
    mbe_stage_kernel<<<(n + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK, WARPS_PER_BLOCK * 32, stream_kernel_smem(), ctx->stream>>>(
        STAGE_TONE, n, base + pbytes + ibytes, (uint32_t*)base, nullptr, nullptr, nullptr, (float*)ctx->d_out[1],
        dstar_id ? (const int32_t*)(base + pbytes) : nullptr, nullptr, ctx->d_tab);
    ctx->launches++;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(cur_parms, base, pbytes, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpyAsync(pcmf, ctx->d_out[1], ob, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int mbe_b200_comfort_noise(mbe_b200_ctx* ctx, int n, uint32_t* rng_words4, float* pcmf) {
    if (!ctx) {
        return MBE_B200_E_ARG;
    }
    if (n < 0 || !rng_words4 || !pcmf) {
        return fail(ctx, MBE_B200_E_ARG, "comfort_noise: bad argument", cudaSuccess);
    }
    if (n == 0) {
        return 0;
    }
    if (check_idle(ctx, "comfort_noise") < 0) {
        return MBE_B200_E_ARG;
    }
    CU(cudaSetDevice(ctx->device));
    const size_t rb = (size_t)n * 16, ob = (size_t)n * NS * 4;
    int rc;
    if ((rc = ensure(ctx, &ctx->d_in, &ctx->d_in_cap, rb)) < 0 || (rc = ensure(ctx, &ctx->d_out[1], &ctx->d_out_cap[1], ob)) < 0) {
        return rc;
    }
    CU(cudaMemcpyAsync(ctx->d_in, rng_words4, rb, cudaMemcpyHostToDevice, ctx->stream));
    mbe_stage_kernel<<<(n + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK, WARPS_PER_BLOCK * 32, stream_kernel_smem(), ctx->stream>>>(
        STAGE_COMFORT, n, nullptr, nullptr, nullptr, nullptr, nullptr, (float*)ctx->d_out[1], nullptr, (uint32_t*)ctx->d_in,
        ctx->d_tab);
    ctx->launches++;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(rng_words4, ctx->d_in, rb, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpyAsync(pcmf, ctx->d_out[1], ob, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int mbe_b200_channel_step(mbe_b200_ctx* ctx, int codec, int step, int n, uint8_t* frames, uint8_t* bits, int32_t* status) {
    if (!ctx) {
        return MBE_B200_E_ARG;
    }
    int fb, pb;
    const bool need_fr = step >= 0 && step <= 2, need_d = step == 2 || step == 3;
    if (mbe_b200_geometry(codec, &fb, &pb) != 0 || step < 0 || step > 3 || (step == 3 && codec != MBE_B200_IMBE7100X4400) || n < 0 ||
        !status || (need_fr && !frames) || (need_d && !bits)) {
        return fail(ctx, MBE_B200_E_ARG, "channel_step: bad argument", cudaSuccess);
    }
    if (n == 0) {
        return 0;
    }
    if (check_idle(ctx, "channel_step") < 0) {
        return MBE_B200_E_ARG;
    }
    CU(cudaSetDevice(ctx->device));
    const size_t fbytes = need_fr ? (size_t)n * fb : 0, dbytes = need_d ? (size_t)n * pb : 0;
    int rc;
    if ((rc = ensure(ctx, &ctx->d_in, &ctx->d_in_cap, fbytes + 16)) < 0 || (rc = ensure(ctx, &ctx->d_out[3], &ctx->d_out_cap[3], dbytes + 16)) < 0 ||
        (rc = ensure(ctx, &ctx->d_out[2], &ctx->d_out_cap[2], (size_t)n * 4)) < 0) {
        return rc;
    }
    if (need_fr) {
        CU(cudaMemcpyAsync(ctx->d_in, frames, fbytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    if (need_d) {
        CU(cudaMemcpyAsync(ctx->d_out[3], bits, dbytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    void (*k)(int, int, uint8_t*, uint8_t*, int32_t*, const DevTables*) =
        codec == 0 ? mbe_front_step_kernel<0> : (codec == 1 ? mbe_front_step_kernel<1> : (codec == 2 ? mbe_front_step_kernel<2> : mbe_front_step_kernel<3>));
    k<<<(n + 7) / 8, 256, 0, ctx->stream>>>(step, n, (uint8_t*)ctx->d_in, (uint8_t*)ctx->d_out[3], (int32_t*)ctx->d_out[2], ctx->d_tab);
    ctx->launches++;
    CU(cudaGetLastError());
    if (step <= 1) {
        CU(cudaMemcpyAsync(frames, ctx->d_in, fbytes, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (need_d) {
        CU(cudaMemcpyAsync(bits, ctx->d_out[3], dbytes, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CU(cudaMemcpyAsync(status, ctx->d_out[2], (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

static int synthesize_speech_impl(mbe_b200_ctx* ctx, int n, void* cur_parms, void* prev_parms, const uint32_t* seeds,
                                  uint32_t* rng_inout, float* pcmf, int16_t* pcm) {
    if (!ctx) {
        return MBE_B200_E_ARG;
    }
    if (n < 0 || !cur_parms || !prev_parms) {
        return fail(ctx, MBE_B200_E_ARG, "synthesize_speech: bad argument", cudaSuccess);
    }
    if (n == 0) {
        return 0;
    }
    if (check_idle(ctx, "synthesize_speech") < 0) {
        return MBE_B200_E_ARG;
    }
    CU(cudaSetDevice(ctx->device));
    const size_t pbytes = (size_t)n * sizeof(Parms);
    const size_t rbytes = rng_inout ? (size_t)n * 16 : (size_t)n * 4;
    int rc;
    // d_in: [cur | prev | seeds or RNG words]
    if ((rc = ensure(ctx, &ctx->d_in, &ctx->d_in_cap, 2 * pbytes + rbytes)) < 0) {
        return rc;
    }
    uint8_t* base = (uint8_t*)ctx->d_in;
    CU(cudaMemcpyAsync(base, cur_parms, pbytes, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(base + pbytes, prev_parms, pbytes, cudaMemcpyHostToDevice, ctx->stream));
    if (rng_inout) {
        CU(cudaMemcpyAsync(base + 2 * pbytes, rng_inout, rbytes, cudaMemcpyHostToDevice, ctx->stream));
    } else if (seeds) {
        CU(cudaMemcpyAsync(base + 2 * pbytes, seeds, rbytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    const size_t ob[2] = {pcm ? (size_t)n * NS * sizeof(int16_t) : 0, pcmf ? (size_t)n * NS * sizeof(float) : 0};
    for (int i = 0; i < 2; ++i) {
        if (ob[i] && (rc = ensure(ctx, &ctx->d_out[i], &ctx->d_out_cap[i], ob[i])) < 0) {
            return rc;
        }
    }
    LaunchArgs a;
    memset(&a, 0, sizeof(a));
    a.mode = MODE_SYNTH;
    a.n_streams = n;
    a.n_frames = 1;
    a.pcm = pcm ? (int16_t*)ctx->d_out[0] : nullptr;
    a.pcmf = pcmf ? (float*)ctx->d_out[1] : nullptr;
    a.tab = ctx->d_tab;
    a.synth_cur = (uint32_t*)base;
    a.synth_prev = (uint32_t*)(base + pbytes);
    a.synth_seeds = (!rng_inout && seeds) ? (const uint32_t*)(base + 2 * pbytes) : nullptr;
    a.synth_rng = rng_inout ? (uint32_t*)(base + 2 * pbytes) : nullptr;
    if ((rc = launch_stream_kernel(ctx, a, ctx->stream)) < 0) {
        return rc;
    }
    CU(cudaMemcpyAsync(cur_parms, base, pbytes, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpyAsync(prev_parms, base + pbytes, pbytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (rng_inout) {
        CU(cudaMemcpyAsync(rng_inout, base + 2 * pbytes, rbytes, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (pcm) {
        CU(cudaMemcpyAsync(pcm, ctx->d_out[0], ob[0], cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (pcmf) {
        CU(cudaMemcpyAsync(pcmf, ctx->d_out[1], ob[1], cudaMemcpyDeviceToHost, ctx->stream));
    }
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int mbe_b200_synthesize_speech(mbe_b200_ctx* ctx, int n, void* cur_parms, void* prev_parms, const uint32_t* seeds,
                               float* pcmf, int16_t* pcm) {
    return synthesize_speech_impl(ctx, n, cur_parms, prev_parms, seeds, nullptr, pcmf, pcm);
}

int mbe_b200_synthesize_speech_rng(mbe_b200_ctx* ctx, int n, void* cur_parms, void* prev_parms, uint32_t* rng_words4,
                                   float* pcmf, int16_t* pcm) {
    if (ctx && !rng_words4) {
        return fail(ctx, MBE_B200_E_ARG, "synthesize_speech_rng: bad argument", cudaSuccess);
    }
    return synthesize_speech_impl(ctx, n, cur_parms, prev_parms, nullptr, rng_words4, pcmf, pcm);
}

int mbe_b200_floattoshort(mbe_b200_ctx* ctx, int n_frames, const float* in, int16_t* out) {
    if (!ctx) {
        return MBE_B200_E_ARG;
    }
    if (n_frames < 0 || !in || !out) {
        return fail(ctx, MBE_B200_E_ARG, "floattoshort: bad argument", cudaSuccess);
    }
    if (n_frames == 0) {
        return 0;
    }
    if (check_idle(ctx, "floattoshort") < 0) {
        return MBE_B200_E_ARG;
    }
    CU(cudaSetDevice(ctx->device));
    const size_t n = (size_t)n_frames * NS;
    int rc;
    if ((rc = ensure(ctx, &ctx->d_in, &ctx->d_in_cap, n * sizeof(float))) < 0) {
        return rc;
    }
    if ((rc = ensure(ctx, &ctx->d_out[0], &ctx->d_out_cap[0], n * sizeof(int16_t))) < 0) {
        return rc;
    }
    CU(cudaMemcpyAsync(ctx->d_in, in, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    if ((rc = mbe_b200_floattoshort_dev(ctx, n_frames, (const float*)ctx->d_in, (int16_t*)ctx->d_out[0], ctx->stream)) < 0) {
        return rc;
    }
    CU(cudaMemcpyAsync(out, ctx->d_out[0], n * sizeof(int16_t), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

}  // extern "C"
