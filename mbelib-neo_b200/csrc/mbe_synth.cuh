// Speech synthesis on one warp: spectral enhancement, adaptive smoothing, noise sources, phase update,
// voiced oscillator bank, FFT/WOLA unvoiced synthesis, tone synthesis, soft clip, float->int16.
// Replaces src/core/mbelib.c:412-1132,1148-1177, src/core/mbe_adaptive.c:116-276,
// src/core/mbe_unvoiced_fft.c:277-761 and the N=256 real radix-4 path of the vendored pffft
// (src/external/pffft/pffft.c:749-926,1109-1196).
//
// The 160 output samples of a frame live in the warp's shared-memory row ws.out: lane i owns samples
// i, 32+i, ..., 128+i.  Rounding-order rules that pin parity with the reference:
//   * per sample, harmonics are added in order l = 1..maxl, previous-frame component before
//     current-frame component (mbelib.c:310-317,1025-1039);
//   * each oscillator is the reference's rotation recurrence, unfused:  c' = c*cd - s*sd,
//     s' = s*cd + c*sd (mbelib.c:213-219), contribution (gain*W[n])*c (mbelib.c:262-265);
//   * FFT butterflies follow FFTPACK radf4/radb4 operation order.
#pragma once
#include "mbe_common.cuh"
#include "mbe_libm.cuh"

namespace mbe {

#ifndef MBE_OSC_UNROLL
#define MBE_OSC_UNROLL 2
#endif
constexpr int kOscUnroll = MBE_OSC_UNROLL;  // oscillator steps per loop body = 4 * kOscUnroll
#define MBE_PI_F 3.14159274101257324f /* (float)M_PI */
// MBE_ABL: timing-only ablation mask for experimental builds (results are wrong when non-zero)
#ifndef MBE_ABL
#define MBE_ABL 0
#endif
#define MBE_CLIP_F ((32767.0f * 0.95f) / 7.0f)

// The glibc-exact transcendental ports are large (double-precision kernels + Payne-Hanek style
// reduction); they are kept out of line so each exists once per kernel image (instruction cache).
__device__ __noinline__ float2 dev_sincosf(float y) {
    float2 r;
    mbelibm::sincosf_glibc(y, &r.x, &r.y);  // x = sin, y = cos
    return r;
}
__device__ __noinline__ float dev_cosf(float y) { return mbelibm::cosf_glibc(y); }
__device__ __noinline__ float dev_sinf(float y) { return mbelibm::sinf_glibc(y); }

__device__ __forceinline__ bool bands_ok(int L) { return L >= 1 && L <= MAXL; }

// ---- whole-struct copies ---------------------------------------------------------------------------
// cur_mp's head (298 words + noiseSeed) lives in shared memory; prev_mp / prev_mp_enhanced keep compact
// subsets there (PrevSmall / EnhSmall); everything else (their remaining head words, and previousUw /
// noiseOverlap of all three) stays in the stream's HBM slot.  Global words are made visible between lanes
// by the __syncwarp() that follows every copy.
// previousUw[256] + noiseOverlap[96] of one struct image to another, both in HBM (11 independent loads per
// lane in flight, then 11 stores)
// (plain pointers: these words are written by this kernel too, so they must not go through the read-only path)
__device__ __forceinline__ void bulk_copy_all(uint32_t* dst, const uint32_t* src, int lane) {
    if (MBE_ABL & 64) {
        return;
    }
    uint32_t v[11];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        v[k] = src[UW_WORD + 32 * k + lane];
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        v[8 + k] = src[OVERLAP_WORD + 32 * k + lane];
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        dst[UW_WORD + 32 * k + lane] = v[k];
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        dst[OVERLAP_WORD + 32 * k + lane] = v[8 + k];
    }
}

// HBM homes of the stream's three structs (651-word mbe_parms images) + a scratch image.
// SPLIT: the frame program runs as two kernels (mbe_split.cuh).  The parameter kernel then owns everything but the
// previousUw arrays: its struct copies move only noiseOverlap and RECORD the copy as a 4-bit op code in the frame's
// descriptor; the synthesis kernel, which owns previousUw, replays the ops in order.
template <bool SPLIT_>
struct StreamHomeT {
    static constexpr bool SPLIT = SPLIT_;
    uint32_t* cur;
    uint32_t* prev;
    uint32_t* enh;
    uint32_t* spill;
};
using StreamHome = StreamHomeT<false>;

enum { OP_CUR_FROM_PREV = 1, OP_PREV_FROM_CUR = 2, OP_ENH_FROM_CUR = 3, OP_CUR_FROM_ENH = 4, OP_ZERO_CUR = 5,
       OP_SPILL_FROM_CUR = 6, OP_CUR_FROM_SPILL = 7, OP_SYNTH = 8 };

__device__ __forceinline__ void record_op(WarpWS& ws, int op, int lane) {
    if (lane == 0) {
        const unsigned n = ws.nops;
        ws.ops |= (n < 8u) ? ((unsigned)op << (4u * n)) : 0u;   // (a frame records at most seven)
        ws.nops = n + 1u;
    }
}

template <class H>
__device__ __forceinline__ void bulk_copy(WarpWS& ws, const H&, uint32_t* dst, const uint32_t* src, int op, int lane) {
    if (H::SPLIT) {
        uint32_t v[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            v[k] = src[OVERLAP_WORD + 32 * k + lane];
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            dst[OVERLAP_WORD + 32 * k + lane] = v[k];
        }
        record_op(ws, op, lane);
    } else {
        bulk_copy_all(dst, src, lane);
    }
}

template <class H>
__device__ __forceinline__ void bulk_zero(WarpWS& ws, const H&, uint32_t* g, int lane) {
    if (!H::SPLIT) {
#pragma unroll
        for (int i = lane; i < 256; i += 32) {
            g[UW_WORD + i] = 0u;
        }
    } else {
        record_op(ws, OP_ZERO_CUR, lane);
    }
#pragma unroll
    for (int i = lane; i < 96; i += 32) {
        g[OVERLAP_WORD + i] = 0u;
    }
}

__device__ __forceinline__ uint32_t* cur_words(WarpWS& ws) { return reinterpret_cast<uint32_t*>(&ws.cur); }
__device__ __forceinline__ int cur_slot(int w) { return w < HEAD_WORDS ? w : HEAD_WORDS; }  // noiseSeed (554) -> 298

template <class H>
__device__ __forceinline__ void prev_from_cur(WarpWS& ws, const H& h, int lane) {
    const uint32_t* c = cur_words(ws);
    uint32_t* p = reinterpret_cast<uint32_t*>(&ws.prev);
#pragma unroll
    for (int j = lane; j < PREV_WORDS; j += 32) {
        p[j] = c[cur_slot(prev_word(j))];
    }
#pragma unroll
    for (int j = lane; j < PREV_HOME_WORDS; j += 32) {
        const int w = prev_home_word(j);
        h.prev[w] = c[w];
    }
    bulk_copy(ws, h, h.prev, h.cur, OP_PREV_FROM_CUR, lane);
    __syncwarp();
}
template <class H>
__device__ __forceinline__ void enh_from_cur(WarpWS& ws, const H& h, int lane, bool bulk = true) {
    const uint32_t* c = cur_words(ws);
    uint32_t* e = reinterpret_cast<uint32_t*>(&ws.enh);
#pragma unroll
    for (int j = lane; j < ENH_WORDS; j += 32) {
        e[j] = c[cur_slot(enh_word(j))];
    }
#pragma unroll
    for (int j = lane; j < ENH_HOME_WORDS; j += 32) {
        h.enh[ENH_HOME_WORD0 + j] = c[ENH_HOME_WORD0 + j];
    }
    if (bulk) {  // (the synthesis stages write prev_mp_enhanced's previousUw / noiseOverlap themselves)
        bulk_copy(ws, h, h.enh, h.cur, OP_ENH_FROM_CUR, lane);
    }
    if (lane == 0) {
        ws.w0row_enh = ws.w0row_prev;  // candidate table row of the fundamental that just became prev_mp_enhanced's
    }
    __syncwarp();
}
template <class H>
__device__ __forceinline__ void cur_from_prev(WarpWS& ws, const H& h, int lane) {
    uint32_t* c = cur_words(ws);
    const uint32_t* p = reinterpret_cast<const uint32_t*>(&ws.prev);
#pragma unroll
    for (int j = lane; j < PREV_WORDS; j += 32) {
        c[cur_slot(prev_word(j))] = p[j];
    }
#pragma unroll
    for (int j = lane; j < PREV_HOME_WORDS; j += 32) {
        const int w = prev_home_word(j);
        c[w] = h.prev[w];
    }
    bulk_copy(ws, h, h.cur, h.prev, OP_CUR_FROM_PREV, lane);
    __syncwarp();
}
template <class H>
__device__ __forceinline__ void cur_from_enh(WarpWS& ws, const H& h, int lane) {
    uint32_t* c = cur_words(ws);
    const uint32_t* e = reinterpret_cast<const uint32_t*>(&ws.enh);
#pragma unroll
    for (int j = lane; j < ENH_WORDS; j += 32) {
        c[cur_slot(enh_word(j))] = e[j];
    }
#pragma unroll
    for (int j = lane; j < ENH_HOME_WORDS; j += 32) {
        c[ENH_HOME_WORD0 + j] = h.enh[ENH_HOME_WORD0 + j];
    }
    bulk_copy(ws, h, h.cur, h.enh, OP_CUR_FROM_ENH, lane);
    __syncwarp();
}

// default model of mbe_initMbeParms / mbe_initAmbeParms_common (head fields + noiseSeed)
template <class P>
__device__ __forceinline__ void fill_default_small(P* p, float w0, int L, int K, float mute_thr, int lane) {
    for (int l = lane; l <= 56; l += 32) {
        p->Ml[l] = 1.0f;
        p->Vl[l] = 0;
        p->log2Ml[l] = 0.0f;
        p->PHIl[l] = 0.0f;
        p->PSIl[l] = 0.0f;
    }
    if (lane == 0) {
        p->swn = 0;
        p->tonePhase = 0;
        p->w0 = w0;
        p->L = L;
        p->K = K;
        p->gamma = 0.0f;
        p->localEnergy = 75000.0f;
        p->amplitudeThreshold = 20480;
        p->errorRate = 0.0f;
        p->errorCountTotal = 0;
        p->errorCount4 = 0;
        p->repeatCount = 0;
        p->mutingThreshold = mute_thr;
        p->noiseSeed = -1.0f;
    }
    __syncwarp();
}

__device__ __forceinline__ void fill_default(Parms* p, float w0, int L, int K, float mute_thr, int lane) {
    fill_default_small(p, w0, L, K, mute_thr, lane);
    for (int i = lane; i < 256; i += 32) {
        p->previousUw[i] = 0.0f;
    }
    for (int i = lane; i < 96; i += 32) {
        p->noiseOverlap[i] = 0.0f;
    }
    __syncwarp();
}

template <class H>
__device__ __noinline__ void init_all(WarpWS& ws, const H& h, float w0, int L, int K, float mute_thr, int lane) {
    fill_default_small(&ws.cur, w0, L, K, mute_thr, lane);
    bulk_zero(ws, h, h.cur, lane);
    __syncwarp();
    prev_from_cur(ws, h, lane);
    enh_from_cur(ws, h, lane);
}

__device__ __forceinline__ void zero_out(WarpWS& ws, int lane) {
#pragma unroll
    for (int c = 0; c < 5; ++c) {
        ws.out[32 * c + lane] = 0.0f;
    }
}

// ---- spectral amplitude enhancement (mbelib.c:412-661); returns pre-enhancement Rm0 -------------
// cos(l w0) by the reference's rotation recurrence from one sincosf(w0): one lane's worth of serial work
__device__ __forceinline__ void cos_recurrence(float w0, int L, float* cosl) {
    const float2 sc = dev_sincosf(w0);
    const float ss = sc.x, cs = sc.y;
    float c = 1.0f, s = 0.0f;
#pragma unroll 4
    for (int l = 1; l <= L; ++l) {
        const float cn = (c * cs) - (s * ss);
        const float sn = (s * cs) + (c * ss);
        c = cn;
        s = sn;
        cosl[l] = c;
    }
}

// fills DevTables::cosw at context creation: one thread per row, the same code the frames would run
__global__ void mbe_costab_kernel(DevTables* T) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= COSW_ROWS) {
        return;
    }
    float w0;
    if (r < COSW_A2450) {
        w0 = T->imbe_w0[r - COSW_IMBE];
    } else if (r < COSW_A2450_SILENCE) {
        w0 = T->a2450_w0[r - COSW_A2450];
    } else if (r == COSW_A2450_SILENCE) {
        w0 = T->a2450_w0_silence;
    } else if (r < COSW_A2400_SILENCE) {
        w0 = T->a2400_w0[r - COSW_A2400];
    } else if (r == COSW_A2400_SILENCE) {
        w0 = T->a2400_w0_silence;
    } else if (r == COSW_IMBE_DEFAULT) {
        w0 = T->imbe_default_w0;
    } else {
        w0 = T->ambe_default_w0;
    }
    T->cosw_w0[r] = w0;
    T->cosw[r][0] = 1.0f;
    cos_recurrence(w0, 56, T->cosw[r]);
    for (int l = 0; l <= 56; ++l) {
        T->stepsc[r][l] = dev_sincosf(w0 * (float)l);  // the expression the bank evaluates for harmonic l's step
    }
}

// scratch: 176 floats, 16-byte aligned (the workspace union: the decode scratch is dead, the synthesis has not begun).
// The ordered sums (Rm0, Rm1, sum of M^2; mbelib.c:490-494) run over arrays padded with zeros to a multiple of four
// harmonics (x + 0 = x), four terms per LDS.128.  On return scratch[0..] holds the enhanced magnitudes M_1..M_L, zero
// padded the same way, for the amplitude sum of the adaptive smoothing.
__device__ __forceinline__ float spectral_enhance(WarpWS& ws, const DevTables* T, float* scratch, int lane) {
    ParmsSmall& cur = ws.cur;
    const int L = cur.L;
    if (!bands_ok(L)) {
        return 0.0f;
    }
    const float w0 = cur.w0;
    if (MBE_ABL & 32) {
        return 1000.0f;
    }
    const int Lpad = (L + 3) & ~3;
    // the cosines come from the table when this frame's (or, after a repeat, the previous frame's) row matches w0
    // bit for bit; otherwise (erasure model, imported state, first frame of a launch after a repeat) from the recurrence
    int row = ws.w0row;
    bool hit = row >= 0 && row < COSW_ROWS && __float_as_uint(T->cosw_w0[row]) == __float_as_uint(w0);
    if (!hit) {
        row = ws.w0row_prev;
        hit = row >= 0 && row < COSW_ROWS && __float_as_uint(T->cosw_w0[row]) == __float_as_uint(w0);
    }
    float2* pair = reinterpret_cast<float2*>(scratch);  // (M^2, M^2 cos) of harmonic l at [l - 1]
    float cosv[2] = {0.0f, 0.0f};
    __syncwarp();
    if (hit) {
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int l = 1 + lane + 32 * r;
            if (l <= L) {
                cosv[r] = T->cosw[row][l];
            }
        }
    } else {
        float* cosl = scratch + 2 * 58;
        cos_recurrence(w0, L, cosl);
        __syncwarp();
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int l = 1 + lane + 32 * r;
            if (l <= L) {
                cosv[r] = cosl[l];
            }
        }
        row = -1;
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int l = 1 + lane + 32 * r;
        if (l <= L) {
            const float m = cur.Ml[l];
            const float m2 = m * m;
            pair[l - 1] = make_float2(m2, m2 * cosv[r]);
        } else if (l <= Lpad) {
            pair[l - 1] = make_float2(0.0f, 0.0f);
        }
    }
    if (lane == 0) {
        ws.w0row_prev = (short)row;
    }
    __syncwarp();
    // serial: Rm0 = sum M^2, Rm1 = sum M^2 cos, in harmonic order
    float Rm0 = 0.0f, Rm1 = 0.0f;
    {
        const float4* p4 = reinterpret_cast<const float4*>(scratch);
#pragma unroll 2
        for (int i = 0; i < Lpad; i += 4) {
            const float4 u = p4[i >> 1], v = p4[(i >> 1) + 1];
            Rm0 += u.x;
            Rm1 += u.y;
            Rm0 += u.z;
            Rm1 += u.w;
            Rm0 += v.x;
            Rm1 += v.y;
            Rm0 += v.z;
            Rm1 += v.w;
        }
    }
    const float R2m0 = Rm0 * Rm0;
    const float R2m1 = Rm1 * Rm1;
    __syncwarp();
    float Mv[2] = {0.0f, 0.0f};
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int l = 1 + lane + 32 * r;
        if (l <= L) {
            float M = cur.Ml[l];
            if (M != 0.0f) {
                const float cosw = cosv[r];
                float W = sqrtf(M)
                          * sqrtf(sqrtf(((0.96f * MBE_PI_F) * ((R2m0 + R2m1) - ((2.0f * Rm0) * Rm1 * cosw)))
                                        / ((w0 * Rm0) * (R2m0 - R2m1))));
                if ((8 * l) <= L) {
                } else if (W > 1.2f) {
                    M = 1.2f * M;
                } else if (W < 0.5f) {
                    M = 0.5f * M;
                } else {
                    M = W * M;
                }
            }
            Mv[r] = M;
            scratch[l - 1] = M * M;  // (the reference squares |M|: same product)
        } else if (l <= Lpad) {
            scratch[l - 1] = 0.0f;
        }
    }
    __syncwarp();
    float sum = 0.0f;
    {
        const float4* p4 = reinterpret_cast<const float4*>(scratch);
#pragma unroll 2
        for (int i = 0; i < Lpad; i += 4) {
            const float4 u = p4[i >> 2];
            sum += u.x;
            sum += u.y;
            sum += u.z;
            sum += u.w;
        }
    }
    const float g = (sum == 0.0f) ? 1.0f : sqrtf(Rm0 / sum);
    __syncwarp();
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int l = 1 + lane + 32 * r;
        if (l <= L) {
            const float M = g * Mv[r];
            cur.Ml[l] = M;
            scratch[l - 1] = M;
        }
    }
    __syncwarp();
    return Rm0;
}

// ---- adaptive smoothing, JMBE algorithms #111-116 (mbe_adaptive.c:151-276) -----------------------
// ml_list (may be null): the magnitudes M_1..M_L as spectral_enhance left them, zero padded to a multiple of four
__device__ __forceinline__ void adaptive_smoothing(ParmsSmall& cur, const EnhSmall& prev, int has_rm0, float rm0,
                                                   int lane, const float* ml_list = nullptr) {
    if (!bands_ok(cur.L) || !bands_ok(prev.L)) {
        return;
    }
    const int L = cur.L;
    if (!has_rm0) {
        rm0 = 0.0f;
        for (int l = 1; l <= L; ++l) {
            rm0 += cur.Ml[l] * cur.Ml[l];
        }
    }
    const float rate = cur.errorRate;
    const int etot = cur.errorCountTotal;
    const int e4 = cur.errorCount4;
    float pe = prev.localEnergy;
    if (pe < 10000.0f) {
        pe = 75000.0f;
    }
    float le = 0.95f * pe + 0.05f * rm0;
    if (le < 10000.0f) {
        le = 10000.0f;
    }
    float VM;
    if (rate <= 0.005f && etot <= 4) {
        VM = 3.40282346638528859812e+38f;
    } else {
        float x8 = sqrtf(sqrtf(sqrtf(le)));
        float en = x8 * x8 * x8;
        if (rate <= 0.0125f && e4 == 0) {
            VM = (45.255f * en) / mbelibm::expf_glibc(277.26f * rate, d_exp2_tab);
        } else {
            VM = 1.414f * en;
        }
    }
    int pt = prev.amplitudeThreshold;
    if (pt <= 0) {
        pt = 20480;
    }
    int Tm;
    if (rate <= 0.005f && etot <= 6) {
        Tm = 20480;
    } else {
        Tm = 6000 - (300 * etot) + pt;
    }
    __syncwarp();
    for (int l = 1 + lane; l <= L; l += 32) {
        if (cur.Ml[l] > VM) {
            cur.Vl[l] = 1;
        }
    }
    float Am = 0.0f;
    if (ml_list) {
        const float4* p4 = reinterpret_cast<const float4*>(ml_list);
#pragma unroll 2
        for (int i = 0; i < L; i += 4) {
            const float4 u = p4[i >> 2];
            Am += u.x;
            Am += u.y;
            Am += u.z;
            Am += u.w;
        }
    } else {
#pragma unroll 4
        for (int l = 1; l <= L; ++l) {
            Am += cur.Ml[l];
        }
    }
    __syncwarp();
    if (lane == 0) {
        cur.localEnergy = le;
        cur.amplitudeThreshold = Tm;
    }
    if (Am > (float)Tm && Am > 0.0f) {
        const float sc = (float)Tm / Am;
        for (int l = 1 + lane; l <= L; l += 32) {
            cur.Ml[l] *= sc;
        }
    }
    __syncwarp();
}

// ---- comfort noise (mbe_adaptive.c:116-131): java.util.Random-style LCG, jump-ahead per lane ------
__device__ __noinline__ void comfort_noise(WarpWS& ws, const DevTables* T, int lane) {
    const float gain = (0.003f * 32767.0f) / 7.0f;
    const unsigned long long mask = (1ULL << 48) - 1ULL;
    const unsigned long long s0 = ws.rng.comfort;
    __syncwarp();
#pragma unroll 1
    for (int c = 0; c < 5; ++c) {
        const int i = 32 * c + lane;
        const unsigned long long st = (T->cnA[i + 1] * s0 + T->cnC[i + 1]) & mask;
        const unsigned r24 = (unsigned)(st >> 24);
        const float u = ((float)r24 / 16777216.0f) * 2.0f - 1.0f;
        ws.out[i] = u * gain;
    }
    if (lane == 0) {
        ws.rng.comfort = (T->cnA[160] * s0 + T->cnC[160]) & mask;
    }
    __syncwarp();
}

// ---- white noise with overlap (mbe_unvoiced_fft.c:304-341) --------------------------------------
// noise_peek: the raw samples 1..56 of the frame's buffer (what the phase update reads) come from the
// overlap of the previous buffer, or are zero on a cold start; nothing is advanced yet.
// The two loads are issued early (noise_fetch) and parked in shared memory later (noise_peek) so that their HBM/L2
// latency hides behind the adaptive smoothing.
__device__ __forceinline__ float2 noise_fetch(const WarpWS& ws, const float* cur_overlap, int lane) {
    const bool cold = ws.cur.noiseSeed < 0.0f;
    float2 v;
    v.x = cold ? 0.0f : cur_overlap[lane];
    v.y = (cold || lane + 32 >= 57) ? 0.0f : cur_overlap[lane + 32];
    return v;
}
__device__ __forceinline__ void noise_peek(WarpWS& ws, float2 v, int lane) {
    ws.u.nz[lane] = v.x;
    if (lane + 32 < 57) {
        ws.u.nz[lane + 32] = v.y;
    }
    __syncwarp();
}

// unvoiced-noise LCG x -> (171 x + 11213) mod 53125 (mbe_unvoiced_fft.c:277-302): coefficients of k steps at once
__host__ __device__ constexpr unsigned lcg_pow_a(int k) {
    unsigned long long a = 1;
    for (int i = 0; i < k; ++i) {
        a = (171ull * a) % 53125ull;
    }
    return (unsigned)a;
}
__host__ __device__ constexpr unsigned lcg_pow_c(int k) {
    unsigned long long c = 0;
    for (int i = 0; i < k; ++i) {
        c = (171ull * c + 11213ull) % 53125ull;
    }
    return (unsigned)c;
}

// make_noise: builds the frame's 256-sample buffer, advances the LCG / overlap state and writes the
// WINDOWED buffer (noise * W256) straight into the FFT input.  cur_overlap = cur_mp->noiseOverlap in HBM.
// enh_overlap (may be null): prev_mp_enhanced->noiseOverlap gets the same new tail right away, which saves the
// HBM -> HBM copy of the struct hand-over after synthesis.
__device__ __forceinline__ void make_noise(WarpWS& ws, float* cur_overlap, float* enh_overlap, const DevTables* T,
                                           const BlockTables* bt, int lane) {
    ParmsSmall& cur = ws.cur;
    float* A = ws.u.fft.a;
    const float seed = cur.noiseSeed;
    if (seed < 0.0f) {
        for (int i = lane; i < NFFT; i += 32) {
            A[i] = 0.0f;  // 0 * window
        }
        for (int i = lane; i < 96; i += 32) {
            cur_overlap[i] = 0.0f;
            if (enh_overlap) {
                enh_overlap[i] = 0.0f;
            }
        }
        const float ns = ws.rng.uv_override ? (float)ws.rng.uv_seed : 3147.0f;
        __syncwarp();
        if (lane == 0) {
            cur.noiseSeed = ns;
            ws.rng.uv_override = 0;  // the override is consumed by the first cold start only
        }
        __syncwarp();
        return;
    }
    // x_{32c + lane} = jump_lane(x_{32c}); x_{32(c+1)} = jump_32(x_{32c}); the frame leaves the generator at x_160
    constexpr unsigned A32 = lcg_pow_a(32), C32 = lcg_pow_c(32);
    unsigned sc = ((unsigned)seed) % 53125u;
    const uint2 jl = bt->uv_jump[lane];
    float ov[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        ov[r] = cur_overlap[32 * r + lane];
    }
#pragma unroll
    for (int c = 0; c < 5; ++c) {
        const int i = 32 * c + lane;
        const unsigned st = (jl.x * sc + jl.y) % 53125u;
        sc = (A32 * sc + C32) % 53125u;
        const float v = (float)st;
        A[96 + i] = v * bt->uvwin[96 + i];
        if (i >= 64) {
            cur_overlap[i - 64] = v;  // overlap <- buffer[160..255] (same lane that read element i - 64 above)
            if (enh_overlap) {
                enh_overlap[i - 64] = v;
            }
        }
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const int i = 32 * r + lane;
        A[i] = ov[r] * bt->uvwin[i];
    }
    const unsigned stn = sc;
    __syncwarp();
    if (lane == 0) {
        cur.noiseSeed = (float)stn;
    }
    __syncwarp();
}

// ---- 256-point real FFT: FFTPACK radix-4 passes (pffft.c:749-926), lanes over butterflies ---------
// Arithmetic (operation order inside every butterfly) is FFTPACK's radf4 / radb4; only the placement of the
// intermediate arrays in shared memory is ours.  The (re, im) pairs (i-1, i) that the ido > 1 butterflies
// read and write are kept 8-byte aligned by shifting those arrays one word, so they move as LDS.64 / STS.64
// and every pass touches shared memory (nearly) conflict-free:
//   X0  time samples, natural order                         phys = p
//   X1  after the ido=1 pass:  [4k + j]                      phys = p                (STS.128 / LDS.128 per k)
//   X2  after the ido=4 pass:  [i + 4j + 16k]  row k, col c  phys = 20*k + c + 1     (rows padded to 20 words)
//   X3  after the ido=16 pass: [i + 16j + 64k] row k, col c  phys = 80*k + c + 1     (rows padded to 80 words)
//   X4  spectrum, FFTPACK order [DC, Re1, Im1, ..., Nyq]     phys = p + 1            (Re_b, Im_b at 2b, 2b+1)
// The backward passes walk the same layouts in reverse.  A and B are the two 324-word ping-pong buffers.
constexpr int X2S = 20, X3S = 80;

struct Cpx { float re, im; };
__device__ __forceinline__ Cpx ld2(const float* p) {
    const float2 v = *reinterpret_cast<const float2*>(p);
    Cpx c = {v.x, v.y};
    return c;
}
__device__ __forceinline__ void st2(float* p, float a, float b) { *reinterpret_cast<float2*>(p) = make_float2(a, b); }

// radf4 inner butterfly for one (i-1, i) pair (pffft.c radf4_ps, the i-loop): x0..x3 = inputs j = 0..3,
// w1..w3 = (wa[i-2], wa[i-1]).  Outputs: o0 = (i-1, i) of output row 0, o2 = (i-1, i) of row 2,
// m3 = (ic-1, ic) of row 3, m1 = (ic-1, ic) of row 1.
__device__ __forceinline__ void radf4_pair(Cpx x0, Cpx x1, Cpx x2, Cpx x3, Cpx w1, Cpx w2, Cpx w3, Cpx& o0, Cpx& m1, Cpx& o2,
                                           Cpx& m3) {
    float cr2 = x1.re, ci2 = x1.im, cr3 = x2.re, ci3 = x2.im, cr4 = x3.re, ci4 = x3.im;
    float t;
    t = cr2 * w1.im;
    cr2 = (cr2 * w1.re) + (ci2 * w1.im);
    ci2 = (ci2 * w1.re) - t;
    t = cr3 * w2.im;
    cr3 = (cr3 * w2.re) + (ci3 * w2.im);
    ci3 = (ci3 * w2.re) - t;
    t = cr4 * w3.im;
    cr4 = (cr4 * w3.re) + (ci4 * w3.im);
    ci4 = (ci4 * w3.re) - t;
    const float tr1 = cr2 + cr4, tr4 = cr4 - cr2;
    const float tr2 = x0.re + cr3, tr3 = x0.re - cr3;
    const float ti1 = ci2 + ci4, ti4 = ci2 - ci4;
    const float ti2 = x0.im + ci3, ti3 = x0.im - ci3;
    o0.re = tr1 + tr2;
    m3.re = tr2 - tr1;
    o2.re = ti4 + tr3;
    m1.re = tr3 - ti4;
    o0.im = ti1 + ti2;
    m3.im = ti1 - ti2;
    o2.im = tr4 + ti3;
    m1.im = tr4 - ti3;
}
// radf4, i = 0 column: a0..a3 = inputs j = 0..3 -> (0,0) (ido-1,1) (0,2) (ido-1,3)
__device__ __forceinline__ void radf4_first(float a0, float a1, float a2, float a3, float& o00, float& oL1, float& o02,
                                            float& oL3) {
    const float tr1 = a1 + a3;
    const float tr2 = a0 + a2;
    oL1 = a0 - a2;
    o02 = a3 - a1;
    o00 = tr1 + tr2;
    oL3 = tr2 - tr1;
}
// radf4, i = ido-1 column: inputs j = 0..3 -> (ido-1,0) (0,1) (ido-1,2) (0,3)
__device__ __forceinline__ void radf4_last(float c, float a, float d, float b, float& oL0, float& o01, float& oL2,
                                           float& o03) {
    const float nhs2 = -0.70710678118654752440f;
    const float ti1 = nhs2 * (a + b);
    const float tr1 = nhs2 * (b - a);
    oL0 = tr1 + c;
    oL2 = c - tr1;
    o01 = ti1 - d;
    o03 = ti1 + d;
}

// radb4 inner butterfly: p0 = (i-1, i) of input row 0, p2 = of row 2, q3 = (ic-1, ic) of row 3, q1 = of row 1;
// outputs y0..y3 = (i-1, i) of output j = 0..3
__device__ __forceinline__ void radb4_pair(Cpx p0, Cpx q1, Cpx p2, Cpx q3, Cpx w1, Cpx w2, Cpx w3, Cpx& y0, Cpx& y1, Cpx& y2,
                                           Cpx& y3) {
    const float tr1 = p0.re - q3.re;
    const float tr2 = p0.re + q3.re;
    const float ti4 = p2.re - q1.re;
    const float tr3 = p2.re + q1.re;
    y0.re = tr2 + tr3;
    float cr3 = tr2 - tr3;
    const float ti3 = p2.im - q1.im;
    const float tr4 = p2.im + q1.im;
    float cr2 = tr1 - tr4;
    float cr4 = tr1 + tr4;
    const float ti1 = p0.im + q3.im;
    const float ti2 = p0.im - q3.im;
    y0.im = ti2 + ti3;
    float ci3 = ti2 - ti3;
    float ci2 = ti1 + ti4;
    float ci4 = ti1 - ti4;
    float t;
    t = cr2 * w1.im;
    y1.re = (cr2 * w1.re) - (ci2 * w1.im);
    y1.im = (ci2 * w1.re) + t;
    t = cr3 * w2.im;
    y2.re = (cr3 * w2.re) - (ci3 * w2.im);
    y2.im = (ci3 * w2.re) + t;
    t = cr4 * w3.im;
    y3.re = (cr4 * w3.re) - (ci4 * w3.im);
    y3.im = (ci4 * w3.re) + t;
}
// radb4, i = 0 column: a = (0,0) d = (ido-1,1) c = (0,2) b = (ido-1,3) -> outputs j = 0..3
__device__ __forceinline__ void radb4_first(float a, float d, float c, float b, float& y0, float& y1, float& y2, float& y3) {
    const float tr3 = 2.f * d;
    const float tr2 = a + b;
    const float tr1 = a - b;
    const float tr4 = 2.f * c;
    y0 = tr2 + tr3;
    y2 = tr2 - tr3;
    y1 = tr1 - tr4;
    y3 = tr1 + tr4;
}
// radb4, i = ido-1 column: c = (ido-1,0) a = (0,1) d = (ido-1,2) b = (0,3) -> outputs j = 0..3
__device__ __forceinline__ void radb4_last(float c, float a, float d, float b, float& y0, float& y1, float& y2, float& y3) {
    const float nsq2 = -1.41421356237309504880f;
    const float tr1 = c - d;
    const float tr2 = c + d;
    const float ti1 = b + a;
    const float ti2 = b - a;
    y0 = tr2 + tr2;
    y1 = nsq2 * (ti1 - tr1);
    y2 = ti2 + ti2;
    y3 = nsq2 * (ti1 + tr1);
}

// forward transform: A = X0 on entry, A = X4 on exit (B scratch).  tw = FFTPACK twiddle table:
// ido=64 rows at 0/64/128, ido=16 rows at 192/208/224, ido=4 rows at 240/244/248.
__device__ __forceinline__ void rfft256_forward_inl(float* __restrict__ A, float* __restrict__ B, const float* __restrict__ tw,
                                                    int lane) {
    // ---- ido = 1, l1 = 64: X0 -> X1
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int k = lane + 32 * h;
        float4 o;
        radf4_first(A[k], A[k + 64], A[k + 128], A[k + 192], o.x, o.y, o.z, o.w);
        *reinterpret_cast<float4*>(B + 4 * k) = o;
    }
    __syncwarp();
    // ---- ido = 4, l1 = 16: X1 -> X2, lane = k owns row k
    if (lane < 16) {
        const float4 v0 = *reinterpret_cast<const float4*>(B + 4 * lane);
        const float4 v1 = *reinterpret_cast<const float4*>(B + 4 * lane + 64);
        const float4 v2 = *reinterpret_cast<const float4*>(B + 4 * lane + 128);
        const float4 v3 = *reinterpret_cast<const float4*>(B + 4 * lane + 192);
        float c0, c7, c8, c15, c3, c4, c11, c12;
        radf4_first(v0.x, v1.x, v2.x, v3.x, c0, c7, c8, c15);
        radf4_last(v0.w, v1.w, v2.w, v3.w, c3, c4, c11, c12);
        Cpx o0, m1, o2, m3;
        const Cpx x0 = {v0.y, v0.z}, x1 = {v1.y, v1.z}, x2 = {v2.y, v2.z}, x3 = {v3.y, v3.z};
        radf4_pair(x0, x1, x2, x3, ld2(tw + 240), ld2(tw + 244), ld2(tw + 248), o0, m1, o2, m3);
        float* row = A + X2S * lane;
        row[1] = c0;
        st2(row + 2, o0.re, o0.im);
        *reinterpret_cast<float4*>(row + 4) = make_float4(c3, c4, m1.re, m1.im);
        *reinterpret_cast<float4*>(row + 8) = make_float4(c7, c8, o2.re, o2.im);
        *reinterpret_cast<float4*>(row + 12) = make_float4(c11, c12, m3.re, m3.im);
        row[16] = c15;
    }
    __syncwarp();
    // ---- ido = 16, l1 = 4: X2 -> X3, lane = 8k + q: q >= 1 pair (2q-1, 2q), q == 0 the two edge columns
    {
        const int k = lane >> 3, q = lane & 7;
        const float* in = A + X2S * k;     // rows k + 4j
        float* out = B + X3S * k;
        if (q) {
            Cpx o0, m1, o2, m3;
            radf4_pair(ld2(in + 2 * q), ld2(in + 4 * X2S + 2 * q), ld2(in + 8 * X2S + 2 * q), ld2(in + 12 * X2S + 2 * q),
                       ld2(tw + 190 + 2 * q), ld2(tw + 206 + 2 * q), ld2(tw + 222 + 2 * q), o0, m1, o2, m3);
            st2(out + 2 * q, o0.re, o0.im);
            st2(out + 32 - 2 * q, m1.re, m1.im);
            st2(out + 32 + 2 * q, o2.re, o2.im);
            st2(out + 64 - 2 * q, m3.re, m3.im);
        } else {
            float o00, oL1, o02, oL3, oL0, o01, oL2, o03;
            radf4_first(in[1], in[4 * X2S + 1], in[8 * X2S + 1], in[12 * X2S + 1], o00, oL1, o02, oL3);
            radf4_last(in[16], in[4 * X2S + 16], in[8 * X2S + 16], in[12 * X2S + 16], oL0, o01, oL2, o03);
            out[1] = o00;
            st2(out + 16, oL0, o01);
            st2(out + 32, oL1, o02);
            st2(out + 48, oL2, o03);
            out[64] = oL3;
        }
    }
    __syncwarp();
    // ---- ido = 64, l1 = 1: X3 -> X4, lane p >= 1 pair (2p-1, 2p), lane 0 the two edge columns
    if (lane) {
        const int p2 = 2 * lane;
        Cpx o0, m1, o2, m3;
        radf4_pair(ld2(B + p2), ld2(B + X3S + p2), ld2(B + 2 * X3S + p2), ld2(B + 3 * X3S + p2), ld2(tw + p2 - 2),
                   ld2(tw + 62 + p2), ld2(tw + 126 + p2), o0, m1, o2, m3);
        st2(A + p2, o0.re, o0.im);
        st2(A + 128 - p2, m1.re, m1.im);
        st2(A + 128 + p2, o2.re, o2.im);
        st2(A + 256 - p2, m3.re, m3.im);
    } else {
        float o00, oL1, o02, oL3, oL0, o01, oL2, o03;
        radf4_first(B[1], B[X3S + 1], B[2 * X3S + 1], B[3 * X3S + 1], o00, oL1, o02, oL3);
        radf4_last(B[64], B[X3S + 64], B[2 * X3S + 64], B[3 * X3S + 64], oL0, o01, oL2, o03);
        A[1] = o00;
        st2(A + 64, oL0, o01);
        st2(A + 128, oL1, o02);
        st2(A + 192, oL2, o03);
        A[256] = oL3;
    }
    __syncwarp();
}
__device__ __noinline__ void rfft256_forward(float* __restrict__ A, float* __restrict__ B, const float* __restrict__ tw,
                                             int lane) {
    rfft256_forward_inl(A, B, tw, lane);
}

// backward transform: A = X4 on entry (unscaled spectrum; every bin is multiplied by scale[bin] as it is
// loaded, mbe_unvoiced_fft.c:688-712), A = X0 on exit (B scratch)
__device__ __noinline__ void rfft256_backward(float* __restrict__ A, float* __restrict__ B, const float* __restrict__ tw,
                                              const float* __restrict__ scale, int lane) {
    // ---- ido = 64: X4 -> X3
    if (lane) {
        const int p2 = 2 * lane;
        Cpx p0 = ld2(A + p2), q1 = ld2(A + 128 - p2), pp2 = ld2(A + 128 + p2), q3 = ld2(A + 256 - p2);
        const float s0 = scale[lane], s1 = scale[64 - lane], s2 = scale[64 + lane], s3 = scale[128 - lane];
        p0.re *= s0;
        p0.im *= s0;
        q1.re *= s1;
        q1.im *= s1;
        pp2.re *= s2;
        pp2.im *= s2;
        q3.re *= s3;
        q3.im *= s3;
        Cpx y0, y1, y2, y3;
        radb4_pair(p0, q1, pp2, q3, ld2(tw + p2 - 2), ld2(tw + 62 + p2), ld2(tw + 126 + p2), y0, y1, y2, y3);
        st2(B + p2, y0.re, y0.im);
        st2(B + X3S + p2, y1.re, y1.im);
        st2(B + 2 * X3S + p2, y2.re, y2.im);
        st2(B + 3 * X3S + p2, y3.re, y3.im);
    } else {
        const float s0 = scale[0], s32 = scale[32], s64 = scale[64], s96 = scale[96], s128 = scale[128];
        float y0, y1, y2, y3;
        radb4_first(A[1] * s0, A[128] * s64, A[129] * s64, A[256] * s128, y0, y1, y2, y3);
        B[1] = y0;
        B[X3S + 1] = y1;
        B[2 * X3S + 1] = y2;
        B[3 * X3S + 1] = y3;
        radb4_last(A[64] * s32, A[65] * s32, A[192] * s96, A[193] * s96, y0, y1, y2, y3);
        B[64] = y0;
        B[X3S + 64] = y1;
        B[2 * X3S + 64] = y2;
        B[3 * X3S + 64] = y3;
    }
    __syncwarp();
    // ---- ido = 16: X3 -> X2
    {
        const int k = lane >> 3, q = lane & 7;
        const float* in = B + X3S * k;
        float* out = A + X2S * k;
        if (q) {
            Cpx y0, y1, y2, y3;
            radb4_pair(ld2(in + 2 * q), ld2(in + 32 - 2 * q), ld2(in + 32 + 2 * q), ld2(in + 64 - 2 * q), ld2(tw + 190 + 2 * q),
                       ld2(tw + 206 + 2 * q), ld2(tw + 222 + 2 * q), y0, y1, y2, y3);
            st2(out + 2 * q, y0.re, y0.im);
            st2(out + 4 * X2S + 2 * q, y1.re, y1.im);
            st2(out + 8 * X2S + 2 * q, y2.re, y2.im);
            st2(out + 12 * X2S + 2 * q, y3.re, y3.im);
        } else {
            float y0, y1, y2, y3;
            radb4_first(in[1], in[32], in[33], in[64], y0, y1, y2, y3);
            out[1] = y0;
            out[4 * X2S + 1] = y1;
            out[8 * X2S + 1] = y2;
            out[12 * X2S + 1] = y3;
            radb4_last(in[16], in[17], in[48], in[49], y0, y1, y2, y3);
            out[16] = y0;
            out[4 * X2S + 16] = y1;
            out[8 * X2S + 16] = y2;
            out[12 * X2S + 16] = y3;
        }
    }
    __syncwarp();
    // ---- ido = 4: X2 -> X1, lane = k owns row k
    if (lane < 16) {
        const float* row = A + X2S * lane;
        const float c0 = row[1];
        const Cpx p0 = ld2(row + 2);
        const float4 r1 = *reinterpret_cast<const float4*>(row + 4);    // cols 3..6
        const float4 r2 = *reinterpret_cast<const float4*>(row + 8);    // cols 7..10
        const float4 r3 = *reinterpret_cast<const float4*>(row + 12);   // cols 11..14
        const float c15 = row[16];
        float f0, f1, f2, f3, l0, l1, l2, l3;
        radb4_first(c0, r2.x, r2.y, c15, f0, f1, f2, f3);
        radb4_last(r1.x, r1.y, r3.x, r3.y, l0, l1, l2, l3);
        const Cpx q1 = {r1.z, r1.w}, pp2 = {r2.z, r2.w}, q3 = {r3.z, r3.w};
        Cpx y0, y1, y2, y3;
        radb4_pair(p0, q1, pp2, q3, ld2(tw + 240), ld2(tw + 244), ld2(tw + 248), y0, y1, y2, y3);
        *reinterpret_cast<float4*>(B + 4 * lane) = make_float4(f0, y0.re, y0.im, l0);
        *reinterpret_cast<float4*>(B + 4 * lane + 64) = make_float4(f1, y1.re, y1.im, l1);
        *reinterpret_cast<float4*>(B + 4 * lane + 128) = make_float4(f2, y2.re, y2.im, l2);
        *reinterpret_cast<float4*>(B + 4 * lane + 192) = make_float4(f3, y3.re, y3.im, l3);
    }
    __syncwarp();
    // ---- ido = 1: X1 -> X0
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int k = lane + 32 * h;
        const float4 v = *reinterpret_cast<const float4*>(B + 4 * k);
        float y0, y1, y2, y3;
        radb4_first(v.x, v.y, v.z, v.w, y0, y1, y2, y3);
        A[k] = y0;
        A[k + 64] = y1;
        A[k + 128] = y2;
        A[k + 192] = y3;
    }
    __syncwarp();
}

// ---- unvoiced synthesis (mbe_unvoiced_fft.c:714-761); adds into ws.out and writes cur.previousUw --
// ws.u.fft.a holds the windowed noise on entry; enh_uw = prev_mp_enhanced->previousUw in HBM.  The spectrum
// stays in FFTPACK's native order (the reference's "ordered" layout is only a permutation of it).
// Three stages (the stream kernel may put a block barrier between them to keep its warps on the same code):
//   unvoiced_analyse   forward transform;   unvoiced_shape   band scales + backward transform;
//   unvoiced_overlap   weighted overlap-add into ws.out, hand-over of the block to cur_mp->previousUw
__device__ __forceinline__ void unvoiced_analyse(WarpWS& ws, const BlockTables* bt, int lane) {
    float* scale = ws.u.fft.scale;
    for (int i = lane; i < 129; i += 32) {
        scale[i] = 0.0f;
    }
    if (!(MBE_ABL & 128)) {
        rfft256_forward(ws.u.fft.a, ws.u.fft.b, bt->tw, lane);   // ends with __syncwarp: scale[] zeros are visible too
    }
}

__device__ __forceinline__ void unvoiced_shape(WarpWS& ws, const BlockTables* bt, int lane) {
    ParmsSmall& cur = ws.cur;
    float* A = ws.u.fft.a;
    float* scale = ws.u.fft.scale;
    const int L = cur.L;
    const float mult = (256.0f / (2.0f * 3.14159265358979323846f)) * cur.w0;
    for (int l = 1 + lane; l <= L; l += 32) {
        int a = (int)ceilf((l - 0.5f) * mult);
        int b = (int)ceilf((l + 0.5f) * mult);
        if (a < 0) {
            a = 0;
        }
        if (b > NFFT / 2) {
            b = NFFT / 2;
        }
        if (cur.Vl[l] == 0 && b > a) {
            float num = 0.0f;
            int s = a;
            if (s == 0) {
                num += A[1] * A[1];
                s = 1;
            }
            for (int bin = s; bin < b; ++bin) {
                const Cpx v = ld2(A + 2 * bin);
                num += (v.re * v.re) + (v.im * v.im);
            }
            if (num > 1e-10f) {
                const float sc = 146.17696f * cur.Ml[l] / sqrtf(num / (float)(b - a));
                for (int bin = a; bin < b; ++bin) {
                    scale[bin] = sc;
                }
            }
        }
    }
    __syncwarp();
    // per-bin scaling happens inside the backward transform; bin 128 (Nyquist) is never covered by a band
    if (!(MBE_ABL & 128)) {
        rfft256_backward(A, ws.u.fft.b, bt->tw, scale, lane);
    }
}

// wola_fetch: the previous frame's tail prev_mp_enhanced->previousUw[128..255], fetched before the backward
// transform so that the loads are back when the overlap-add needs them
struct WolaTail { float ps[4]; };
__device__ __forceinline__ WolaTail wola_fetch(const float* enh_uw, int lane) {
    WolaTail t;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        t.ps[c] = enh_uw[128 + 32 * c + lane];
    }
    return t;
}

// enh_uw_out (may be null): prev_mp_enhanced->previousUw receives the new block together with cur_mp->previousUw
__device__ __forceinline__ void unvoiced_overlap(WarpWS& ws, float* cur_uw, float* enh_uw_out, const WolaTail& tail,
                                                 const BlockTables* bt, int lane) {
    const float* A = ws.u.fft.a;
    const float inv = 1.0f / (float)NFFT;
    // weighted overlap-add of this frame's block (scaled by 1/N as it is read) with the previous frame's,
    // then the soft clip (mbelib.c:669-689)
#pragma unroll
    for (int c = 0; c < 5; ++c) {
        const int n = 32 * c + lane;
        const float den = bt->wola_den[n];
        const float ps = (c < 4) ? tail.ps[c < 4 ? c : 0] : 0.0f;
        const float cs = (n - 32 >= 0) ? (A[n - 32] * inv) : 0.0f;
        float v = ws.out[n];
        if (den > 1e-10f) {
            v += ((bt->wola_wp[n] * ps) + (bt->wola_wc[n] * cs)) / den;
        }
        if (v > MBE_CLIP_F) {
            v = MBE_CLIP_F;
        } else if (v < -MBE_CLIP_F) {
            v = -MBE_CLIP_F;
        }
        ws.out[n] = v;
    }
    // hand the block to the state
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const float v = A[32 * c + lane] * inv;
        cur_uw[32 * c + lane] = v;
        if (enh_uw_out) {
            enh_uw_out[32 * c + lane] = v;
        }
    }
    __syncwarp();
}

// ---- voiced oscillator bank (mbelib.c:953-1040) --------------------------------------------------
// kinds: 0 = previous-frame windowed component, 1 = current-frame windowed component,
//        2 = phase/amplitude-interpolated harmonic (l < 8, both voiced, stable pitch)
//
// build_components: the ordered component list of one stream (l ascending, previous before current).
// Windowed components whose gain is exactly zero (the faded bands of mbelib.c:912-929) are dropped:
// their contribution is +-0 and x + (+-0) == x for every accumulator value that can occur.
__device__ __forceinline__ void build_components(WarpWS& ws, int maxl, int lane) {
    const ParmsSmall& cur = ws.cur;
    const EnhSmall& prev = ws.enh;
    const float cw0 = cur.w0, pw0 = prev.w0;
    const bool stable = fabsf(cw0 - pw0) < (0.1f * cw0);
    int ncomp = 0;
    unsigned k2mask = 0;
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int l = 1 + lane + 32 * r;
        bool cv = false, pv = false;
        float gp = 0.0f, gc = 0.0f;
        if (l <= maxl) {
            cv = (cur.Vl[l] == 1);
            pv = (prev.Vl[l] == 1);
            gp = 2.0f * prev.Ml[l];
            gc = 2.0f * cur.Ml[l];
            // keep zero-gain components whose phase is not finite (their product is NaN, not 0)
            if (gp == 0.0f && !isfinite(prev.PHIl[l])) {
                gp = __int_as_float(0x7fc00000);
            }
            if (gc == 0.0f && !isfinite(cur.PHIl[l])) {
                gc = __int_as_float(0x7fc00000);
            }
        }
        const bool interp = (l < 8) && cv && pv && stable;
        const bool first = interp || (pv && gp != 0.0f);   // first slot of this harmonic
        const bool second = cv && !interp && gc != 0.0f;   // second slot
        const unsigned mf = __ballot_sync(FULL, first);
        const unsigned ms = __ballot_sync(FULL, second);
        const unsigned lt = (1u << lane) - 1u;
        int idx = ncomp + __popc(mf & lt) + __popc(ms & lt);
        if (r == 0) {
            // interpolated harmonics have l < 8, so their list positions are < 14
            k2mask = __reduce_or_sync(FULL, interp ? (1u << idx) : 0u);
        }
        if (first) {
            ws.comp[idx] = (unsigned char)((l << 2) | (interp ? 2 : 0));
            idx++;
        }
        if (second) {
            ws.comp[idx] = (unsigned char)((l << 2) | 1);
        }
        ncomp += __popc(mf) + __popc(ms);
    }
    if (lane == 0) {
        ws.ncomp = ncomp;
        ws.k2mask = k2mask;
    }
    __syncwarp();
}

// publish_components: a stream tells the block how many oscillator slots it needs this frame and appends its
// phase-interpolated harmonics to the block's work list (any order: every item writes its own tile column).
__device__ __forceinline__ void publish_components(BlockShared* bs, int parity, const WarpWS& ws, int go, int warp, int lane) {
    if (lane == 0) {
        bs->cnt[parity][warp] = go ? ws.ncomp : 0;
    }
    const unsigned m = go ? ws.k2mask : 0u;
    if (m) {
        const int n = __popc(m);
        int at = 0;
        if (lane == 0) {
            at = atomicAdd(&bs->n_interp[parity], n);
        }
        at = __shfl_sync(FULL, at, 0);
        if (lane < n) {
            // the item's per-sample phase increment (mbelib.c:959-961) is the same for all 160 samples: computed once here,
            // one lane per item, instead of once per 32-sample chunk by whoever renders it
            const int pos = (int)__fns(m, 0, lane + 1);
            const int l = ws.comp[pos] >> 2;
            const float cw0 = ws.cur.w0, pw0 = ws.enh.w0;
            const float pw0l = pw0 * (float)l;
            const float dphi = ws.cur.PHIl[l] - ws.enh.PHIl[l] - (((pw0 + cw0) * (float)(l * NS)) / 2.0f);
            const float dw = (1.0f / (float)NS)
                             * (dphi - (2.0f * MBE_PI_F * floorf((dphi + MBE_PI_F) / (2.0f * MBE_PI_F))));
            bs->interp[parity][at + lane] = (unsigned short)((warp << 8) | pos);
            bs->interp_a1[parity][at + lane] = pw0l + dw;
        }
    }
}

// Oscillator tile: 32 samples x 32 slots, no padding.  Slot column c of sample row n lives at
// n*32 + (c ^ ((n & 7) << 2)): phase A (lane = slot, one row per store) and phase B (lane = sample, LDS.128 over
// four consecutive slots) are both bank-conflict free.
__device__ __forceinline__ int tile_at(int n, int c) { return n * 32 + (c ^ ((n & 7) << 2)); }

// voiced_bank_block: ALL warps of the block call this once per frame (block barriers inside).
// The component lists of the block's streams are laid end to end (each stream's start rounded up to a
// multiple of four slots) and cut into passes of 32 slots; pass p of a round is run by warp p:
//   phase A  lane = slot: the lane runs that component's oscillator 32 steps (the reference's unfused
//            rotation recurrence) and writes the finished contribution (gain*W[n])*cos into its warp's
//            tile[n][lane]; the phase-interpolated harmonics of the round (one cosf per sample) are
//            dealt round-robin to all warps, lane = sample;
//   phase B  lane = sample, warp = stream: adds its stream's slots in list order (LDS.128, four adds
//            each) from whichever tiles they landed in.
// So oscillator work is spread evenly over the block no matter how the components are distributed
// over streams, and a stream's additions keep the reference's order.
__device__ __forceinline__ void voiced_bank_block(WarpWS* wsa, BlockShared* bs, int parity, const BlockTables* bt,
                                                  const DevTables* T, StageTimer& tm, int warp, int lane) {
    constexpr int W = WARPS_PER_BLOCK;
    static_assert(W <= 16, "owner search and slot offsets are sized for at most 16 streams per block");
    WarpWS& me = wsa[warp];
    const int* cnt = bs->cnt[parity];
    const int n_interp = bs->n_interp[parity];
    const unsigned short* interp = bs->interp[parity];
    const float* interp_a1 = bs->interp_a1[parity];
    if (warp == 0 && lane == 0) {
        bs->n_interp[parity ^ 1] = 0;  // next frame's list (its appends come after at least one more block barrier)
    }
    // slot offsets: exclusive prefix of the counts, each rounded up to a multiple of four (every warp
    // keeps its own copy in shared memory; lanes 0..W-1 scan)
    {
        const int padded = (lane < W) ? ((cnt[lane] + 3) & ~3) : 0;
        int incl = padded;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int up = __shfl_up_sync(FULL, incl, d);
            if (lane >= d) {
                incl += up;
            }
        }
        if (lane <= W) {
            me.off[lane] = (unsigned short)(incl - padded);  // lane W: total
        } else if (lane < W + 3) {
            me.off[lane] = 0xffffu;                          // sentinels for the owner search
        }
        __syncwarp();
    }
    const unsigned short* off = me.off;
    const int total = off[W];
    if (total == 0) {
        return;
    }
    const int my_lo = off[warp], my_cnt = cnt[warp];
    const int my_hi = my_lo + ((my_cnt + 3) & ~3);
    float* tile = me.u.tile;
    float* tcol[8];  // this lane's (= slot's) column in tile rows n = m (mod 8): tile_at(n, lane) = 32 n + (lane ^ 4m)
#pragma unroll
    for (int m = 0; m < 8; ++m) {
        tcol[m] = tile + (lane ^ (m << 2));
    }

#pragma unroll 1
    for (int base = 0; base < total; base += 32 * W) {
        // ---- oscillator owned by this lane in this round (idle slots and interpolated ones write zeros)
        const int k = base + 32 * warp + lane;
        // owner = the last stream whose first slot is <= k (offsets are non-decreasing; empty streams share theirs
        // with the next one), found by a branch-free binary search over the 16 offset entries
        int owner = 0;
        owner += (off[owner + 8] <= k) ? 8 : 0;
        owner += (off[owner + 4] <= k) ? 4 : 0;
        owner += (off[owner + 2] <= k) ? 2 : 0;
        owner += (off[owner + 1] <= k) ? 1 : 0;
        int j = k - off[owner];
        if (owner >= W || j >= cnt[owner]) {
            owner = -1;
            j = 0;
        }
        float g = 0.f, c = 0.f, s = 0.f, cd = 0.f, sd = 0.f;
        const float* Wb = bt->voiced_win;
        bool k2lane = false;  // this lane's slot is an interpolated harmonic: written by whoever computes it
        if (owner >= 0) {
            const WarpWS& o = wsa[owner];
            const int id = o.comp[j];
            if ((id & 3) == 2) {
                k2lane = true;
            } else {
                const int l = id >> 2;
                float step, ph, w0;
                int row;
                if ((id & 3) == 0) {
                    w0 = o.enh.w0;
                    row = o.w0row_enh;
                    step = w0 * (float)l;
                    ph = o.enh.PHIl[l];
                    g = 2.0f * o.enh.Ml[l];
                    Wb = bt->voiced_win + WIN_PREV;
                } else {
                    w0 = o.cur.w0;
                    row = o.w0row_prev;   // (after the enhancement: the row that matched this frame's fundamental)
                    step = w0 * (float)l;
                    ph = o.cur.PHIl[l] - (step * (float)NS);
                    g = 2.0f * o.cur.Ml[l];
                }
                // sincosf(l w0) from the device-generated table when the row's fundamental is this one bit for bit; the two
                // loads do not depend on each other and are in flight while the phase's sincosf runs
                const bool rowok = row >= 0 && row < COSW_ROWS;
                const int rr = rowok ? row : 0;
                const float tw0 = T->cosw_w0[rr];
                float2 d = T->stepsc[rr][l];
                const float2 p = (MBE_ABL & 4) ? make_float2(ph, step) : dev_sincosf(ph);
                if (!(rowok && __float_as_uint(tw0) == __float_as_uint(w0))) {
                    d = dev_sincosf(step);
                }
                sd = d.x;
                cd = d.y;
                s = p.x;
                c = p.y;
            }
        }
        STAGE_T(8);  // offsets + oscillator start states
        // this stream's slots inside the round
        const int lo = max(my_lo, base), hi = min(my_hi, base + 32 * W);
        // interpolated harmonics of the round (one cosf per sample, about a fifth of an oscillator pass each): warps
        // without a pass in the first round take up to three each, the rest is dealt round-robin to everybody
        int n_mine = 0;
        {
            auto take = [&](int t) {
                const int item = interp[t];
                const int slot = off[item >> 8] + (item & 255);
                if (slot >= base && slot < base + 32 * W) {
                    if (lane == 0) {
                        me.interp_item[n_mine] = (unsigned short)t;  // index into the block's work list
                    }
                    ++n_mine;
                }
            };
            const int npass0 = min(W, (total + 31) >> 5);
            const int n_idle = W - npass0;
            const int first_end = min(n_interp, 3 * n_idle);
            if (warp >= npass0) {
                for (int t = warp - npass0; t < first_end; t += n_idle) {
                    take(t);
                }
            }
            for (int t = first_end + warp; t < n_interp; t += W) {
                take(t);
            }
        }
        __syncwarp();
        const bool has_pass = (base + 32 * warp) < total;  // warps beyond the last slot skip phase A
#pragma unroll 1
        for (int ch = 0; ch < 5; ++ch) {
            const float* Wc = Wb + 32 * ch;
            if (has_pass && !(MBE_ABL & 2)) {
                // 32 oscillator steps, fully unrolled: row n of the tile is written at tcol[n & 7] + 32 n
#pragma unroll
                for (int n4 = 0; n4 < 8; ++n4) {
                    const float4 w4 = *reinterpret_cast<const float4*>(Wc + 4 * n4);
                    const float wv[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int n = 4 * n4 + q;
                        if (!k2lane) {
                            tcol[n & 7][32 * n] = (g * wv[q]) * c;
                        }
                        const float cn = (c * cd) - (s * sd);
                        const float sn = (s * cd) + (c * sd);
                        c = cn;
                        s = sn;
                    }
                }
            }
            STAGE_T(9);  // phase A
            if (n_mine && !(MBE_ABL & 8)) {
                const int n = 32 * ch + lane;
#pragma unroll 1
                for (int q = 0; q < n_mine; ++q) {
                    const int t = me.interp_item[q];
                    const int item = interp[t];
                    const int i = item >> 8, pos = item & 255;
                    const WarpWS& o = wsa[i];
                    const int slot = off[i] + pos - base;  // slot index inside the round
                    const int l = o.comp[pos] >> 2;
                    const float cw0 = o.cur.w0, pw0 = o.enh.w0;
                    const float th = o.enh.PHIl[l] + (interp_a1[t] * (float)n)
                                     + (((cw0 - pw0) * (float)(l * n * n)) / (float)(2 * NS));
                    const float am = o.enh.Ml[l] + (((float)n / (float)NS) * (o.cur.Ml[l] - o.enh.Ml[l]));
                    wsa[slot >> 5].u.tile[tile_at(lane, slot & 31)] = 2.0f * am * dev_cosf(th);
                }
            }
            STAGE_T(10);  // interpolated harmonics
            if (!(MBE_ABL & 512)) {  // (512: timing-only bound on what the bank's barriers cost; results are wrong)
                __syncthreads();
            }
            STAGE_T(11);  // wait for phase A of the block
            if (hi > lo && !(MBE_ABL & 1)) {
                const int n = 32 * ch + lane;
                float a = me.out[n];
                int k4 = lo - base;
                const int end = hi - base;
#pragma unroll 1
                while (k4 < end) {
                    // the part of this stream's slot range that lies in one tile: loads first, then the adds in order
                    const int tix = k4 >> 5;
                    const int e = min(end, (tix + 1) << 5);
                    // row `lane` of that tile; its four-slot groups sit at group ^ (lane & 7)
                    const float4* row = reinterpret_cast<const float4*>(wsa[tix].u.tile + lane * 32);
                    const int sw = lane & 7;
                    int gq = (k4 & 31) >> 2;
                    const int ge = gq + ((e - k4) >> 2);
#pragma unroll 1
                    for (; gq + 4 <= ge; gq += 4) {
                        const float4 v0 = row[gq ^ sw], v1 = row[(gq + 1) ^ sw], v2 = row[(gq + 2) ^ sw], v3 = row[(gq + 3) ^ sw];
                        a += v0.x; a += v0.y; a += v0.z; a += v0.w;
                        a += v1.x; a += v1.y; a += v1.z; a += v1.w;
                        a += v2.x; a += v2.y; a += v2.z; a += v2.w;
                        a += v3.x; a += v3.y; a += v3.z; a += v3.w;
                    }
#pragma unroll 1
                    for (; gq < ge; ++gq) {
                        const float4 v = row[gq ^ sw];
                        a += v.x; a += v.y; a += v.z; a += v.w;
                    }
                    k4 = e;
                }
                me.out[n] = a;
            }
            STAGE_T(12);  // phase B
            if (!(MBE_ABL & 512)) {
                __syncthreads();
            }
            STAGE_T(13);  // wait for phase B of the block
        }
    }
}

// ---- mbe_synthesizeSpeechCore (mbelib.c:1042-1105), split around the block-cooperative voiced bank ----
// cur = ws.cur, prev = ws.enh; the 160 float samples end up in ws.out.
// synth_begin: everything up to the component list.  Returns 1 when the frame continues through
// voiced_bank_block + synth_finish, 0 when it is already complete (silence or comfort noise).
// COMPONENTS = false (split path): the synthesis kernel builds its own component lists from the frame's descriptor
template <bool COMPONENTS = true>
__device__ __noinline__ int synth_begin(WarpWS& ws, const float* cur_overlap, const DevTables* T, int has_rm0,
                                        float rm0, int lane) {
    ParmsSmall& cur = ws.cur;
    EnhSmall& prev = ws.enh;
    zero_out(ws, lane);
    if (!bands_ok(cur.L) || !bands_ok(prev.L)) {
        __syncwarp();
        return 0;  // silence
    }
    const float2 nz01 = noise_fetch(ws, cur_overlap, lane);
    adaptive_smoothing(cur, prev, has_rm0, rm0, lane, has_rm0 ? reinterpret_cast<const float*>(&ws.u) : nullptr);

    const bool mute_on_rate = fabsf(cur.mutingThreshold - 0.096f) > 1e-6f;
    if (cur.repeatCount >= 4 || (mute_on_rate && cur.errorRate > cur.mutingThreshold)) {
        comfort_noise(ws, T, lane);
        __syncwarp();
        return 0;
    }
    noise_peek(ws, nz01, lane);

    // bands present in only one frame fade as zero-amplitude voiced bands (mbelib.c:912-929)
    int maxl;
    const int cL = cur.L, pL = prev.L;
    if (cL > pL) {
        maxl = cL;
        for (int l = pL + 1 + lane; l <= maxl; l += 32) {
            prev.Ml[l] = 0.0f;
            prev.Vl[l] = 1;
        }
    } else {
        maxl = pL;
        for (int l = cL + 1 + lane; l <= maxl; l += 32) {
            cur.Ml[l] = 0.0f;
            cur.Vl[l] = 1;
        }
    }
    __syncwarp();

    // numUv counts index 0 as well (mbelib.c:902-910)
    int numUv = 0;
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int l = lane + 32 * r;
        const bool uv = (l <= cL) && (cur.Vl[l] == 0);
        numUv += __popc(__ballot_sync(FULL, uv));
    }

    // phase update for all 56 harmonics (mbelib.c:931-951)
    const float cw0 = cur.w0, pw0 = prev.w0;
    const float two_pi = 2.0f * MBE_PI_F;
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int l = 1 + lane + 32 * r;
        if (l <= 56) {
            float wrapped = fmodf(prev.PSIl[l], two_pi);
            if (wrapped < 0.0f) {
                wrapped += two_pi;
            }
            prev.PSIl[l] = wrapped;
            const float psi = wrapped + ((pw0 + cw0) * ((float)(l * NS) / 2.0f));
            cur.PSIl[l] = psi;
            if (l <= (cL / 4)) {
                cur.PHIl[l] = psi;
            } else {
                const float pl = ((2.0f * MBE_PI_F / 53125.0f) * ws.u.nz[l]) - MBE_PI_F;
                cur.PHIl[l] = psi + (((float)numUv * pl) / (float)cL);
            }
        }
    }
    __syncwarp();
    if (COMPONENTS) {
        build_components(ws, maxl, lane);
    } else if (lane == 0) {
        ws.ncomp = maxl;   // split path: what the descriptor carries instead of a component count
    }
    return 1;
}

// synth_finish_*: unvoiced FFT/WOLA synthesis on top of the voiced samples and the soft clip, in three stages.
// enh_home_out: the stream's prev_mp_enhanced image when it is about to become a copy of cur_mp (stream kernel), null
// when the caller keeps its previous-frame blob (batched mbe_synthesizeSpeech).
__device__ __noinline__ void synth_finish_a(WarpWS& ws, uint32_t* cur_home, uint32_t* enh_home_out, const DevTables* T,
                                            const BlockTables* bt, int lane) {
    make_noise(ws, reinterpret_cast<float*>(cur_home + OVERLAP_WORD),
               enh_home_out ? reinterpret_cast<float*>(enh_home_out + OVERLAP_WORD) : nullptr, T, bt, lane);
    unvoiced_analyse(ws, bt, lane);
}
__device__ __forceinline__ WolaTail synth_finish_b(WarpWS& ws, const uint32_t* enh_home, const BlockTables* bt, int lane) {
    const WolaTail tail = wola_fetch(reinterpret_cast<const float*>(enh_home + UW_WORD), lane);
    unvoiced_shape(ws, bt, lane);
    return tail;
}
__device__ __forceinline__ void synth_finish_c(WarpWS& ws, uint32_t* cur_home, uint32_t* enh_home_out, const WolaTail& tail,
                                               const BlockTables* bt, int lane) {
    unvoiced_overlap(ws, reinterpret_cast<float*>(cur_home + UW_WORD),
                     enh_home_out ? reinterpret_cast<float*>(enh_home_out + UW_WORD) : nullptr, tail, bt, lane);
}

// ---- tone synthesis (mbelib.c:692-856, src/internal/mbe_tone.h) -----------------------------------
// dual-tone (DTMF / call-progress) frequency pairs for tone ids 128..163 (src/internal/mbe_tone.h)
static __device__ const unsigned short k_dual_tones[36][2] = {
    {1336, 941}, {1209, 697}, {1336, 697}, {1477, 697}, {1209, 770}, {1336, 770}, {1477, 770}, {1209, 852},
    {1336, 852}, {1477, 852}, {1633, 697}, {1633, 770}, {1633, 852}, {1633, 941}, {1209, 941}, {1477, 941},
    {1162, 820}, {1052, 606}, {1162, 606}, {1279, 606}, {1052, 672}, {1162, 672}, {1279, 672}, {1052, 743},
    {1162, 743}, {1279, 743}, {1430, 606}, {1430, 672}, {1430, 743}, {1430, 820}, {1052, 820}, {1279, 820},
    {440, 350},  {480, 440},  {620, 480},  {490, 350}};

__device__ __forceinline__ bool tone_freqs(int id, float* f1, float* f2) {
    *f1 = *f2 = 0.0f;
    if (id == 5) {
        *f1 = *f2 = 156.25f;
        return true;
    }
    if (id == 6) {
        *f1 = *f2 = 187.5f;
        return true;
    }
    if (id >= 7 && id <= 122) {
        *f1 = *f2 = 31.25f * (float)id;
        return true;
    }
    if (id >= 128 && id <= 163) {
        *f1 = (float)k_dual_tones[id - 128][0];
        *f2 = (float)k_dual_tones[id - 128][1];
        return true;
    }
    return false;
}

__device__ __forceinline__ unsigned tone_step(double hz) {
    double st = (hz / 8000.0) * 4294967296.0;
    return st <= 0.0 ? 0u : (unsigned)(st + 0.5);
}

__device__ __forceinline__ float tone_sample(unsigned phase) {
    const double rad_per_tick = (2.0 * 3.14159265358979323846) / 4294967296.0;
    float ang = (float)(((double)phase * rad_per_tick) - (3.14159265358979323846 / 2.0));
    return dev_sinf(ang);
}

__device__ __noinline__ void render_tone(WarpWS& ws, float f1, float f2, int amp, int lane) {
    ParmsSmall& cur = ws.cur;
    if (f1 <= 0.0f) {
        zero_out(ws, lane);
        __syncwarp();
        return;
    }
    const bool dual = (f2 > 0.0f) && (fabsf(f2 - f1) > 1e-6f);
    const float gain = (((amp < 0) ? 0.0f : (float)amp) / 127.0f) * MBE_CLIP_F;
    const unsigned s1 = tone_step((double)f1);
    const unsigned s2 = dual ? tone_step((double)f2) : 0u;
    const unsigned p1 = (unsigned)cur.swn, p2 = cur.tonePhase;
    __syncwarp();
#pragma unroll 1
    for (int c = 0; c < 5; ++c) {
        const unsigned n1 = (unsigned)(32 * c + lane + 1);
        const float a = tone_sample(p1 + n1 * s1);
        if (dual) {
            const float b = tone_sample(p2 + n1 * s2);
            ws.out[32 * c + lane] = (0.5f * gain * a) + (0.5f * gain * b);
        } else {
            ws.out[32 * c + lane] = gain * a;
        }
    }
    if (lane == 0) {
        cur.swn = (int)(p1 + 160u * s1);
        cur.tonePhase = p2 + 160u * s2;
    }
    __syncwarp();
}

// mbe_floattoshort (mbelib.c:1148-1177,1312-1320): x7, clip to 95 % full scale, truncate
__device__ __forceinline__ short float_to_short(float x) {
    const float maxa = 32767.0f * 0.95f;
    const unsigned u = __float_as_uint(x);
    const unsigned a = u & 0x7fffffffu;
    float v;
    if (a > 0x7f800000u) {
        v = 0.0f;
    } else if (a == 0x7f800000u) {
        v = (u >> 31) ? -maxa : maxa;
    } else {
        v = 7.0f * x;
        if (v > maxa) {
            v = maxa;
        } else if (v < -maxa) {
            v = -maxa;
        }
    }
    return (short)(int)v;
}

}  // namespace mbe
