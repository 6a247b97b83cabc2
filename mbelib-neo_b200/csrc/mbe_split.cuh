// The frame program as THREE kernels (DESIGN 4.5):
//
//   parameter kernel   mbe_stream_kernel<CODEC, SOFT, MODE, /*SPLIT=*/true>: everything that is serial per stream - ECC,
//                      parameter decode, state machine, enhancement, smoothing, phase update, noise-generator state, the
//                      start state of every oscillator - and the frames that need no speech synthesis (silence, tones,
//                      comfort noise).  For every frame it writes a DESCRIPTOR: what the synthesis needs and nothing else.
//                      Its blocks walk their streams in lockstep like the fused kernel's (the program is ~85 KB of SASS;
//                      warps on the same code share their instruction fetches).
//   bank kernel        mbe_split_bank_kernel: the voiced oscillator bank (mbelib.c:953-1040) and nothing else - a loop of a
//                      few hundred instructions that stays in the instruction cache, so its warps need no lockstep: a warp
//                      lays the components of the frames it visits end to end and runs them in 32-slot passes over its
//                      private 32 x 32 tile, a pass crossing frame boundaries freely (phase A: lane = slot runs the
//                      reference's unfused rotation recurrence; phase B: lane = sample adds each frame's slots in the
//                      reference's order).  One warp's latency-bound ordered sums overlap another
//                      warp's FP32-dense recurrences, and a frame with many harmonics delays nobody else.
//   unvoiced kernel    mbe_split_unvoiced_kernel: 256-point FFT / IFFT unvoiced synthesis with weighted overlap-add
//                      (mbe_unvoiced_fft.c:714-761), soft clip, float -> int16.  It owns the previousUw arrays of the
//                      stream's three parameter sets and replays the struct copies the state machine asked for (4-bit op
//                      codes in the descriptor).  Every frame costs the same here, so its blocks run in lockstep for free.
//
// Why three: a first two-kernel cut (one synthesis kernel with decoupled warps, 59 KB of SASS) spent 51 % of its issue
// slots waiting for instructions (profiles/experiments/r02i_*): warps that are not on the same code cannot share fetches,
// and the straight-line transforms are far larger than the 32 KB L1.5 instruction cache.
#pragma once
#include "mbe_common.cuh"
#include "mbe_synth.cuh"

namespace mbe {

// ---- frame descriptor (words) --------------------------------------------------------------------------------------
constexpr int D_OPS = 0;     // previousUw ops of the frame, 4 bits each, in order (OP_*; OP_SYNTH = the synthesis itself)
constexpr int D_INFO = 1;    // bit 0: frame runs the synthesis; bits 8..15 cur L; bits 16..23 oscillator slots (components)
constexpr int D_CW0 = 2;     // cur_mp->w0
constexpr int D_DW0 = 3;     // cur_mp->w0 - prev_mp_enhanced->w0 (the chirp term of the interpolated harmonics)
constexpr int D_SEED = 4;    // cur_mp->noiseSeed before the frame's noise buffer is built (< 0: cold start)
constexpr int D_CU = 6;      // 2 words: bit l-1 = (cur Vl[l] == 0), l = 1..56, after smoothing
constexpr int D_CML = 16;    // cur Ml[1..56]
constexpr int D_OV = 72;     // cur_mp->noiseOverlap[96] before the frame
constexpr int D_KIND = 168;  // 112 bytes: per slot harmonic << 2 | kind (0 previous-frame window, 1 current-frame window,
                             // 2 phase / amplitude interpolated), list order = the reference's summation order
constexpr int D_G = 196;     // per slot, 112 words each: gain            | interpolated: phase increment per sample
constexpr int D_C = 308;     //                           cos(start phase) |               prev PHIl[l]
constexpr int D_S = 420;     //                           sin(start phase) |               prev Ml[l]
constexpr int D_CD = 532;    //                           cos(l w0)        |               cur Ml[l]
constexpr int D_SD = 644;    //                           sin(l w0)
constexpr int D_VOICED = D_G;  // the bank kernel leaves the frame's 160 voiced samples here (its slot records are dead by then)
constexpr int DESC_WORDS = 768;
static_assert(D_SD + 112 <= DESC_WORDS && D_VOICED + NS <= D_S, "descriptor layout");

#ifndef MBE_BWARPS
#define MBE_BWARPS 8
#endif
#ifndef MBE_BMINB
#define MBE_BMINB 4
#endif
#ifndef MBE_UWARPS
#define MBE_UWARPS 8
#endif
#ifndef MBE_UMINB
#define MBE_UMINB 4
#endif
#ifndef MBE_U_LOCKSTEP
#define MBE_U_LOCKSTEP 0
#endif
constexpr int B_WARPS = MBE_BWARPS;   // warps per block of the bank kernel
constexpr int B_MINB = MBE_BMINB;
constexpr int U_WARPS = MBE_UWARPS;   // warps (= streams) per block of the unvoiced kernel
constexpr int U_MINB = MBE_UMINB;

// ---- parameter-kernel side -----------------------------------------------------------------------------------------
// make_noise without the FFT input: advances the generator (seed, overlap of cur_mp and prev_mp_enhanced) exactly like
// make_noise and hands back what the synthesis kernel needs to rebuild the frame's buffer: the overlap and the seed as they
// were before (mbe_unvoiced_fft.c:304-341)
__device__ __forceinline__ void make_noise_state(WarpWS& ws, float* cur_overlap, float* enh_overlap, const BlockTables* bt,
                                                 int lane, float ov[3], float* seed_before) {
    ParmsSmall& cur = ws.cur;
    const float seed = cur.noiseSeed;
    *seed_before = seed;
    if (seed < 0.0f) {
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            ov[r] = 0.0f;
            cur_overlap[32 * r + lane] = 0.0f;
            enh_overlap[32 * r + lane] = 0.0f;
        }
        const float ns = ws.rng.uv_override ? (float)ws.rng.uv_seed : 3147.0f;
        __syncwarp();
        if (lane == 0) {
            cur.noiseSeed = ns;
            ws.rng.uv_override = 0;
        }
        __syncwarp();
        return;
    }
    constexpr unsigned A32 = lcg_pow_a(32), C32 = lcg_pow_c(32);
    constexpr unsigned A64 = lcg_pow_a(64), C64 = lcg_pow_c(64);
    unsigned sc = ((unsigned)seed) % 53125u;
    const uint2 jl = bt->uv_jump[lane];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        ov[r] = cur_overlap[32 * r + lane];
    }
    sc = (A64 * sc + C64) % 53125u;   // the first 64 new samples never reach the overlap
#pragma unroll
    for (int c = 2; c < 5; ++c) {
        const unsigned st = (jl.x * sc + jl.y) % 53125u;
        sc = (A32 * sc + C32) % 53125u;
        const float v = (float)st;
        cur_overlap[32 * (c - 2) + lane] = v;
        enh_overlap[32 * (c - 2) + lane] = v;
    }
    const unsigned stn = sc;
    __syncwarp();
    if (lane == 0) {
        cur.noiseSeed = (float)stn;
    }
    __syncwarp();
}

// the arrays of a synthesis frame's descriptor (after synth_begin: phases updated, lengths reconciled, component list
// built): what the unvoiced kernel reads, and one record per oscillator slot - the start state the fused kernel's bank
// computes per lane (voiced_bank_block), here once, by the kernel that runs in lockstep anyway
__device__ __forceinline__ void emit_desc_arrays(uint32_t* d, const WarpWS& ws, const float ov[3], const DevTables* T,
                                                 int lane) {
    const ParmsSmall& cur = ws.cur;
    const EnhSmall& prev = ws.enh;
    unsigned cu[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int l = 1 + lane + 32 * r;
        int cvl = 2;
        if (l <= 56) {
            cvl = cur.Vl[l];
            d[D_CML + l - 1] = __float_as_uint(cur.Ml[l]);
        }
        cu[r] = __ballot_sync(FULL, cvl == 0);
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        d[D_OV + 32 * r + lane] = __float_as_uint(ov[r]);
    }
    if (lane < 2) {
        d[D_CU + lane] = lane ? cu[1] : cu[0];
    }
    const int ncomp = ws.ncomp;
    const float cw0 = cur.w0, pw0 = prev.w0;
    unsigned char* kinds = reinterpret_cast<unsigned char*>(d + D_KIND);
#pragma unroll 1
    for (int k = lane; k < ncomp; k += 32) {
        const int id = ws.comp[k];
        const int l = id >> 2;
        float g, c, s, cd, sd = 0.0f;
        if ((id & 3) == 2) {
            const float pw0l = pw0 * (float)l;
            const float dphi = cur.PHIl[l] - prev.PHIl[l] - (((pw0 + cw0) * (float)(l * NS)) / 2.0f);
            const float dw = (1.0f / (float)NS) * (dphi - (2.0f * MBE_PI_F * floorf((dphi + MBE_PI_F) / (2.0f * MBE_PI_F))));
            g = pw0l + dw;
            c = prev.PHIl[l];
            s = prev.Ml[l];
            cd = cur.Ml[l];
        } else {
            float step, ph, w0;
            int row;
            if ((id & 3) == 0) {
                w0 = pw0;
                row = ws.w0row_enh;
                step = w0 * (float)l;
                ph = prev.PHIl[l];
                g = 2.0f * prev.Ml[l];
            } else {
                w0 = cw0;
                row = ws.w0row_prev;   // (after the enhancement: the row that matched this frame's fundamental)
                step = w0 * (float)l;
                ph = cur.PHIl[l] - (step * (float)NS);
                g = 2.0f * cur.Ml[l];
            }
            const bool rowok = row >= 0 && row < COSW_ROWS;
            const int rr = rowok ? row : 0;
            const float tw0 = T->cosw_w0[rr];
            float2 dd = T->stepsc[rr][l];
            const float2 p = dev_sincosf(ph);
            if (!(rowok && __float_as_uint(tw0) == __float_as_uint(w0))) {
                dd = dev_sincosf(step);
            }
            sd = dd.x;
            cd = dd.y;
            s = p.x;
            c = p.y;
        }
        kinds[k] = (unsigned char)id;
        d[D_G + k] = __float_as_uint(g);
        d[D_C + k] = __float_as_uint(c);
        d[D_S + k] = __float_as_uint(s);
        d[D_CD + k] = __float_as_uint(cd);
        d[D_SD + k] = __float_as_uint(sd);
    }
    __syncwarp();   // the frame's hand-over rewrites ws.enh: every lane must be done reading it
}

// the descriptor's header; every frame of the launch gets one (a frame without synthesis may still move previousUw).
// emit_desc_info runs BEFORE the frame's hand-over (prev_mp_enhanced <- cur_mp changes w0), emit_desc_ops after it (the
// hand-over may record one more op).
__device__ __forceinline__ void emit_desc_info(uint32_t* d, const WarpWS& ws, int go, float seed_before, int lane) {
    if (lane >= 1 && lane < 5) {
        unsigned v;
        if (lane == 1) {
            v = (go ? 1u : 0u) | ((unsigned)(ws.cur.L & 255) << 8) | ((unsigned)(ws.ncomp & 255) << 16);
        } else if (lane == 2) {
            v = __float_as_uint(ws.cur.w0);
        } else if (lane == 3) {
            v = __float_as_uint(ws.cur.w0 - ws.enh.w0);
        } else {
            v = __float_as_uint(seed_before);
        }
        d[lane] = v;
    }
    __syncwarp();   // (the hand-over that follows rewrites ws.enh)
}
__device__ __forceinline__ void emit_desc_ops(uint32_t* d, const WarpWS& ws, int lane) {
    if (lane == 0) {
        d[D_OPS] = ws.ops;
    }
}

// ---- bank kernel -----------------------------------------------------------------------------------------------------
struct SynthArgs {
    int first_stream, io_base, n_streams, n_frames;
    uint32_t* desc;         // [n_streams][n_frames][DESC_WORDS]
    int16_t* pcm;           // [..][n_frames][160] (frames without synthesis were written by the parameter kernel)
    float* pcmf;
    float pcmf_scale;
    uint32_t* state;        // [max_streams][STATE_WORDS]: only the previousUw words are touched
    const DevTables* tab;
    unsigned long long* counters;   // profiling (may be null): [0] oscillator slots run, [1] of them interpolated harmonics,
                                    // [2] frames synthesised, [3] 32-slot passes of the bank kernel; unvoiced kernel:
                                    // [4] noise spectra taken from the table, [5] noise spectra computed in the kernel
    const int32_t* slots;   // indexed calls: as LaunchArgs (slot_of)
    int slot_base;
    const float* noise_tab; // [NOISE_ROWS][256] forward noise spectra (mbe_noise_table_kernel), null: every frame computes its own
};

// Oscillator tile of the bank kernel: 32 samples x 32 slots, rows padded to 36 words: phase A (lane = slot, one row per
// store) and phase B (lane = sample, LDS.128 over four consecutive slots) are both bank-conflict free, and every access is
// a base register + immediate offset (no swizzle arithmetic in the loops)
constexpr int BT_STRIDE = 36;
#ifndef MBE_BANK_STEPS
#define MBE_BANK_STEPS 16
#endif
constexpr int BANK_STEPS = MBE_BANK_STEPS;   // oscillator steps per loop body of phase A (8 / 16 / 32)
struct __align__(16) BankWS {
    float tile[32 * BT_STRIDE];
    float carry[NS];        // running sums of the frame a pass left open (lane i owns i, 32 + i, ...); 0 while none is
};

// smem: voiced window halves (BlockTables::voiced_win layout, 336 floats) | n / 160 for n = 0..159 | per-warp workspaces
constexpr int BANK_TAB_FLOATS = 336 + NS;

__global__ void __launch_bounds__(B_WARPS * 32, B_MINB) mbe_split_bank_kernel(const SynthArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* vwin = reinterpret_cast<float*>(smem_raw);
    float* nfrac = vwin + 336;   // (float)n / (float)N of the amplitude interpolation (mbelib.c:963), the same division
    BankWS* wsa = reinterpret_cast<BankWS*>(smem_raw + BANK_TAB_FLOATS * sizeof(float));
    for (int i = threadIdx.x; i < 2 * NS; i += blockDim.x) {
        vwin[i < NS ? i : i + (WIN_PREV - NS)] = A.tab->voiced_win[i];
    }
    for (int i = threadIdx.x; i < NS; i += blockDim.x) {
        nfrac[i] = (float)i / (float)NS;
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    BankWS& ws = wsa[warp];
    float* tile = ws.tile;
#pragma unroll
    for (int c = 0; c < 5; ++c) {
        ws.carry[32 * c + lane] = 0.0f;
    }
    // The grid is resident (a few blocks per SM); warp gw visits frames gw, gw + W, gw + 2 W, ... (W warps in the grid).  The
    // oscillator slots of the frames it visits form one queue in visit order, each frame's list padded to a multiple of four
    // (a four-slot group of the tile never straddles frames), and every pass takes the next 32 slots of that queue: only the
    // warp's last pass runs part empty.  Frame sums are independent, so a pass may hold the tail of one frame, whole frames and
    // the head of another; what a frame has summed when a pass ends inside it waits in ws.carry.
    const long long n_items = (long long)A.n_streams * A.n_frames;
    const long long gw = (long long)blockIdx.x * B_WARPS + warp;
    const long long warps_total = (long long)gridDim.x * B_WARPS;
    auto frame_desc = [&](int v) { return A.desc + (size_t)(gw + (long long)v * warps_total) * DESC_WORDS; };

    // The window: frames v0 .. v0 + 31 of the walk, lane j holding frame v0 + j.  Queue positions count from the window's
    // first slot; pos is where the next pass starts.
    int v0 = 0, pos = 0;
    int v_seen = 0;            // frames of the walk before this one were counted and, when they have no slots, zeroed already
    unsigned win = 0u;         // lane j: end of frame j's padded slots in the queue | its slot count << 16 (0 without synthesis)
    int total = 0, n_live = 0; // end of the window's queue; frames of the window that exist
    int n_slots = 0;           // profiling counters (this lane's share of [0]; [1], [2] and [3] are warp-uniform)
    int n_k2 = 0, n_go = 0, n_pass = 0;
    auto load_window = [&]() {
        const long long it = gw + (long long)(v0 + lane) * warps_total;
        const bool live = it < n_items;
        unsigned info = 0u;
        if (live) {
            info = A.desc[(size_t)it * DESC_WORDS + D_INFO];
        }
        const int cnt = (info & 1u) ? (int)((info >> 16) & 255u) : 0;
        int e = (cnt + 3) & ~3;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(FULL, e, d);
            if (lane >= d) {
                e += t;
            }
        }
        win = (unsigned)e | ((unsigned)cnt << 16);
        total = __shfl_sync(FULL, e, 31);
        n_live = __popc(__ballot_sync(FULL, live));
        const bool fresh = (info & 1u) && v0 + lane >= v_seen;
        n_go += __popc(__ballot_sync(FULL, fresh));
        n_slots += fresh ? cnt : 0;
        // a frame that runs the synthesis without a slot still gets its 160 zero samples
        for (unsigned zm = __ballot_sync(FULL, fresh && cnt == 0); zm; zm &= zm - 1u) {
            uint32_t* d = frame_desc(v0 + __ffs(zm) - 1);
#pragma unroll
            for (int c = 0; c < 5; ++c) {
                d[D_VOICED + 32 * c + lane] = 0u;
            }
        }
        v_seen = v0 + 32;
    };
    load_window();
#pragma unroll 1
    while (true) {
        // frames of the window wholly before pos (the next one holds pos); once fewer than 32 slots are left, the window moves
        // on to start at that frame so that the pass can be filled
        const int j0 = __popc(__ballot_sync(FULL, (int)(win & 0xffffu) <= pos));
        if (j0 == 32 && n_live < 32) {
            break;
        }
        if (n_live == 32 && total - pos < 32 && j0 > 0) {
            const int start = __shfl_sync(FULL, (int)(win & 0xffffu), j0 - 1);
            pos = (j0 == 32) ? 0 : pos - start;
            v0 += j0;
            load_window();
            continue;
        }
        ++n_pass;
        // the window frame j that owns queue position pos + lane: the first whose end lies beyond it (31 past the queue's end,
        // where nothing is used)
        const int p = pos + lane;
        int j = 0;
#pragma unroll
        for (int st = 16; st; st >>= 1) {
            if ((int)(__shfl_sync(FULL, win, j + st - 1) & 0xffffu) <= p) {
                j += st;
            }
        }
        const unsigned wj = __shfl_sync(FULL, win, j);
        const int end_j = (int)(wj & 0xffffu), cnt_j = (int)(wj >> 16);
        const int at = p - (end_j - ((cnt_j + 3) & ~3));   // position in frame j's list
        const bool used = at < cnt_j;
        float g = 0.f, c = 0.f, s = 0.f, cd = 0.f, sd = 0.f, dw0 = 0.f;
        int kind = 0, l = 0;
        if (used) {
            const uint32_t* d = frame_desc(v0 + j);
            const unsigned id = reinterpret_cast<const unsigned char*>(d + D_KIND)[at];
            kind = (int)(id & 3u);
            l = (int)(id >> 2);
            g = __uint_as_float(d[D_G + at]);
            c = __uint_as_float(d[D_C + at]);
            s = __uint_as_float(d[D_S + at]);
            cd = __uint_as_float(d[D_CD + at]);
            sd = __uint_as_float(d[D_SD + at]);
            dw0 = __uint_as_float(d[D_DW0]);
        }
        const bool k2lane = (kind == 2);
        const unsigned k2mask = __ballot_sync(FULL, k2lane);
        n_k2 += __popc(k2mask);
        const float* Wb = vwin + ((kind == 0) ? WIN_PREV : 0);
        const float gg = k2lane ? 0.0f : g;   // interpolated slots are written by whoever renders them
        const float rec_c = c, rec_s = s;     // (the recurrence below rotates c and s on every lane)
        // phase B's map of the pass: bit 4g of fchg = the frame changes at four-slot group g; ng groups hold slots; last_open =
        // the frame of the last group has slots beyond this pass.  Every frame but the last one ends inside the pass: all its
        // slots are in registers by now, so its samples may overwrite its slot records
        const int j_up = __shfl_up_sync(FULL, j, 4);
        const unsigned fchg = __ballot_sync(FULL, (lane & 3) == 0 && j != j_up);
        const int ng = min(8, (total - pos) >> 2);
        const bool last_open = ((__ballot_sync(FULL, end_j > pos + 32) >> (4 * (ng - 1))) & 1u) != 0u;
        pos += 32;
#pragma unroll 1
        for (int ch = 0; ch < 5; ++ch) {
            // phase A: 32 oscillator steps, sixteen per loop body (the body stays in the L0 instruction cache)
            const float4* W4 = reinterpret_cast<const float4*>(Wb) + 8 * ch;
            float* tp = tile + lane;
#pragma unroll 1
            for (int h = 0; h < 32 / BANK_STEPS; ++h) {
#pragma unroll
                for (int n4 = 0; n4 < BANK_STEPS / 4; ++n4) {
                    const float4 w4 = W4[(BANK_STEPS / 4) * h + n4];
                    const float wv[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        if (!k2lane) {
                            tp[(4 * n4 + i) * BT_STRIDE] = (gg * wv[i]) * c;   // row n = BANK_STEPS h + 4 n4 + i
                        }
                        const float cn = (c * cd) - (s * sd);
                        const float sn = (s * cd) + (c * sd);
                        c = cn;
                        s = sn;
                    }
                }
                tp += BANK_STEPS * BT_STRIDE;
            }
            // phase-interpolated harmonics of this pass: lane = sample (mbelib.c:953-968); the slot's lane holds its record
            if (k2mask) {
                const int n = 32 * ch + lane;
                const float fn = (float)n, fr = nfrac[n];
                const int nn = n * n;
                for (unsigned m = k2mask; m; m &= m - 1u) {
                    const int sl = __ffs(m) - 1;
                    const float a1 = __shfl_sync(FULL, g, sl), phi = __shfl_sync(FULL, rec_c, sl),
                                pM = __shfl_sync(FULL, rec_s, sl), cM = __shfl_sync(FULL, cd, sl),
                                dw = __shfl_sync(FULL, dw0, sl);
                    const int ll = __shfl_sync(FULL, l, sl);
                    const float th = phi + (a1 * fn) + ((dw * (float)(ll * nn)) / (float)(2 * NS));
                    const float am = pM + (fr * (cM - pM));
                    tile[lane * BT_STRIDE + sl] = 2.0f * am * dev_cosf(th);
                }
            }
            __syncwarp();
            // phase B: lane = sample; the tile's groups in order, each added to the running sum of the frame that owns it
            // (list order = the reference's summation order).  Every sum starts from 0 (pad slots add +0, which is exactly
            // neutral); where the frame changes, the finished frame's samples go straight to its descriptor
            {
                const float4* row = reinterpret_cast<const float4*>(tile + lane * BT_STRIDE);
                float* cr = ws.carry + 32 * ch + lane;
                float a = *cr;
#pragma unroll
                for (int gi = 0; gi < 8; ++gi) {
                    if (gi < ng) {
                        if (gi > 0 && ((fchg >> (4 * gi)) & 1u)) {
                            frame_desc(v0 + __shfl_sync(FULL, j, 4 * gi - 4))[D_VOICED + 32 * ch + lane] = __float_as_uint(a);
                            a = 0.0f;
                        }
                        const float4 v = row[gi];
                        a += v.x;
                        a += v.y;
                        a += v.z;
                        a += v.w;
                    }
                }
                if (!last_open) {
                    frame_desc(v0 + __shfl_sync(FULL, j, 4 * ng - 4))[D_VOICED + 32 * ch + lane] = __float_as_uint(a);
                    a = 0.0f;
                }
                *cr = a;
            }
            __syncwarp();
        }
    }
    if (A.counters) {
        n_slots = __reduce_add_sync(FULL, (unsigned)n_slots);
        if (lane == 0) {
            atomicAdd(&A.counters[0], (unsigned long long)n_slots);
            atomicAdd(&A.counters[1], (unsigned long long)n_k2);
            atomicAdd(&A.counters[2], (unsigned long long)n_go);
            atomicAdd(&A.counters[3], (unsigned long long)n_pass);
        }
    }
}

// ---- unvoiced kernel ---------------------------------------------------------------------------------------------------
// Three transform buffers: a frame runs in two of them (A, B) while the third receives the next frame's noise spectrum from
// the table; the next frame's A is that third buffer, its B the frame's A, and its prefetch target the frame's B.
// With the table, a frame's header words 0..7 and overlap are staged into dstage two frames ahead: the check that picks the
// next frame's table row, and the frame's own ops and noise buffer, wait for no global load.
constexpr int DSTAGE_WORDS = 8 + 96;
struct __align__(16) UnvWS {
    float buf[3][324];
    uint32_t dstage[2][DSTAGE_WORDS];
    float scale[130];
    unsigned n_tab[2];   // frames of the launch whose noise spectrum came from the table / was computed (with A.counters)
};

__device__ __forceinline__ void uw_copy(uint32_t* dst, const uint32_t* src, int lane) {
    uint32_t v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        v[k] = src[UW_WORD + 32 * k + lane];
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        dst[UW_WORD + 32 * k + lane] = v[k];
    }
}

// band scales + backward transform for one frame (unvoiced_shape on descriptor data)
__device__ __forceinline__ void split_unvoiced_shape(UnvWS& ws, float* A, float* B, const uint32_t* d, int L, float w0,
                                                     unsigned cu_lo, unsigned cu_hi, const BlockTables* bt, int lane) {
    float* scale = ws.scale;
    const float mult = (256.0f / (2.0f * 3.14159265358979323846f)) * w0;
    for (int l = 1 + lane; l <= L; l += 32) {
        int a = (int)ceilf((l - 0.5f) * mult);
        int b = (int)ceilf((l + 0.5f) * mult);
        if (a < 0) {
            a = 0;
        }
        if (b > NFFT / 2) {
            b = NFFT / 2;
        }
        const bool uv = ((l <= 32 ? cu_lo >> (l - 1) : cu_hi >> (l - 33)) & 1u) != 0u;
        if (uv && b > a) {
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
                const float sc = 146.17696f * __uint_as_float(d[D_CML + l - 1]) / sqrtf(num / (float)(b - a));
                for (int bin = a; bin < b; ++bin) {
                    scale[bin] = sc;
                }
            }
        }
    }
    __syncwarp();
    rfft256_backward(A, B, bt->tw, scale, lane);
}

// make_noise's FFT input: the windowed 256-sample buffer of a frame whose generator starts at sc (sc < 53125) and whose
// overlap word 32 r + lane is ov[r]
__device__ __forceinline__ void noise_buffer(float* A, unsigned sc, const float ov[3], const BlockTables* bt, int lane) {
    constexpr unsigned A32 = lcg_pow_a(32), C32 = lcg_pow_c(32);
    const uint2 jl = bt->uv_jump[lane];
#pragma unroll
    for (int c = 0; c < 5; ++c) {
        const int i = 32 * c + lane;
        const unsigned st = (jl.x * sc + jl.y) % 53125u;
        sc = (A32 * sc + C32) % 53125u;
        A[96 + i] = (float)st * bt->uvwin[96 + i];
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const int i = 32 * r + lane;
        A[i] = ov[r] * bt->uvwin[i];
    }
}

// the generator state a frame starts from: (unsigned)seed % 53125 for seed >= 0, as make_noise computes it
__device__ __forceinline__ unsigned noise_start(float seed) { return ((unsigned)seed) % 53125u; }

// the frame's windowed noise buffer from its descriptor's seed and overlap words ov[0..95]
__device__ __forceinline__ void split_noise(float* A, float seed, const uint32_t* ov_words, const BlockTables* bt, int lane) {
    if (seed < 0.0f) {
        for (int i = lane; i < NFFT; i += 32) {
            A[i] = 0.0f;
        }
        return;
    }
    float ov[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        ov[r] = __uint_as_float(ov_words[32 * r + lane]);
    }
    noise_buffer(A, noise_start(seed), ov, bt, lane);
}

// ---- noise spectrum table ------------------------------------------------------------------------------------------
// A frame whose overlap is the one its own generator state sc left behind - overlap word k = LCG^(k - 96)(sc), the 96 states
// before sc, which make_noise_state always produces - has a noise buffer that depends on sc alone, and so has its forward
// spectrum.  Row sc of the table is that spectrum, A[1..256] of the X4 layout, computed by the unvoiced kernel's own
// noise_buffer and rfft256_forward.  A frame takes its row only after checking all 96 overlap words bit for bit
// (noise_prefetch); any other frame (cold starts, imported states) computes its own.
constexpr int NOISE_ROWS = 53125;
constexpr int NOISE_TAB_WARPS = 8;

// overlap word 32 r + lane of the natural overlap before generator state sc; bk[r] = (uvBA, uvBC)[32 r + lane]
__device__ __forceinline__ unsigned noise_overlap_word(unsigned sc, uint2 bk) { return (bk.x * sc + bk.y) % 53125u; }

__global__ void __launch_bounds__(NOISE_TAB_WARPS * 32) mbe_noise_table_kernel(const DevTables* __restrict__ T, float* tab) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    BlockTables* bt = reinterpret_cast<BlockTables*>(smem_raw);
    UnvWS* wsa = reinterpret_cast<UnvWS*>(smem_raw + sizeof(BlockTables));
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        bt->tw[i] = T->tw[i];
        bt->uvwin[i] = T->uvwin[i];
    }
    if (threadIdx.x < 32) {
        bt->uv_jump[threadIdx.x] = make_uint2(T->uvA[threadIdx.x], T->uvC[threadIdx.x]);
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    float* A = wsa[warp].buf[0];
    float* B = wsa[warp].buf[1];
#pragma unroll 1
    for (int sc = blockIdx.x * NOISE_TAB_WARPS + warp; sc < NOISE_ROWS; sc += gridDim.x * NOISE_TAB_WARPS) {
        float ov[3];
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const int k = 32 * r + lane;
            ov[r] = (float)noise_overlap_word((unsigned)sc, make_uint2(T->uvBA[k], T->uvBC[k]));
        }
        noise_buffer(A, (unsigned)sc, ov, bt, lane);
        __syncwarp();
        rfft256_forward(A, B, bt->tw, lane);
        float* row = tab + (size_t)sc * NFFT;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            row[32 * q + lane] = A[1 + 32 * q + lane];
        }
        __syncwarp();
    }
}

// 4-byte asynchronous copies global -> shared (the spectrum sits at A + 1, which is 8-byte but not 16-byte aligned)
__device__ __forceinline__ void cp_async4(float* dst, const float* src) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(s), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

// descriptor words 0..7 and the overlap of frame d into a staging buffer (16-byte copies: both runs are 16-byte aligned)
static_assert(D_SEED < 8 && D_INFO < 8 && D_OV % 4 == 0, "staged descriptor words");
__device__ __forceinline__ void stage_desc(uint32_t* st, const uint32_t* d, int lane) {
    if (lane < DSTAGE_WORDS / 4) {
        const int w = 4 * lane;
        const uint32_t* src = d + (w < 8 ? w : D_OV + w - 8);
        const unsigned s = (unsigned)__cvta_generic_to_shared(st + w);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(src) : "memory");
    }
}

// whether a frame's noise spectrum is row sc of the table (st = its staged descriptor words): the frame runs the synthesis,
// seed >= 0, and its overlap is the natural one of sc, word for word (bk = the uvBA / uvBC pairs).  If so, the row is fetched
// into A + 1 (asynchronously: cp_async_wait_all).
__device__ __forceinline__ bool noise_prefetch(const uint32_t* st, const float* tab, const uint2* bk, float* A, int lane) {
    const float seed = __uint_as_float(st[D_SEED]);
    const bool cand = (st[D_INFO] & 1u) && seed >= 0.0f;
    bool ok = cand;
    const unsigned sc = cand ? noise_start(seed) : 0u;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        ok = ok && st[8 + 32 * r + lane] == __float_as_uint((float)noise_overlap_word(sc, bk[32 * r + lane]));
    }
    if (__ballot_sync(FULL, ok) != FULL) {
        return false;
    }
    const float* row = tab + (size_t)sc * NFFT;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        cp_async4(A + 1 + 32 * q + lane, row + 32 * q + lane);
    }
    return true;
}

// one warp = one stream, frames in order (the overlap-add needs the previous frame's block)
__global__ void __launch_bounds__(U_WARPS * 32, U_MINB) mbe_split_unvoiced_kernel(const SynthArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    BlockTables* bt = reinterpret_cast<BlockTables*>(smem_raw);
    uint2* bk = reinterpret_cast<uint2*>(smem_raw + sizeof(BlockTables));   // [96] uvBA / uvBC
    UnvWS* wsa = reinterpret_cast<UnvWS*>(smem_raw + sizeof(BlockTables) + 96 * sizeof(uint2));
    const DevTables* T = A.tab;
    {
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
        for (int i = threadIdx.x; i < 96; i += blockDim.x) {
            bk[i] = make_uint2(T->uvBA[i], T->uvBC[i]);
        }
        __syncthreads();
    }
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    UnvWS& ws = wsa[warp];
    const int s = blockIdx.x * U_WARPS + warp;
    const bool live = s < A.n_streams;
    // (an element an indexed call rejected left descriptors without ops: its slot, possibly out of range, is never used)
    uint32_t* gs = A.state + (size_t)(live ? slot_of(A, s) : A.first_stream) * STATE_WORDS;
    uint32_t* h_cur = gs;
    uint32_t* h_prev = gs + PARMS_WORDS;
    uint32_t* h_enh = gs + 2 * PARMS_WORDS;
    uint32_t* h_spill = gs + SPILL_WORD;
    // bits 0..1: the buffer of the frame's A (see UnvWS); bit 2: its noise spectrum is on its way from the table.  At the top
    // of frame f the warp waits for the copies it issued a frame earlier (frame f's row, frame f + 1's staged words) and
    // issues frame f + 1's row; frame f + 2's words follow once frame f's own staged words have been read.
    unsigned tb = 0u;
    if (live && A.noise_tab) {
        const uint32_t* d0 = A.desc + (size_t)s * A.n_frames * DESC_WORDS;
        stage_desc(ws.dstage[0], d0, lane);
        if (A.n_frames > 1) {
            stage_desc(ws.dstage[1], d0 + DESC_WORDS, lane);
        }
        cp_async_wait_all();
        __syncwarp();
        if (noise_prefetch(ws.dstage[0], A.noise_tab, bk, ws.buf[0], lane)) {
            tb = 4u;
        }
    }
    if (lane == 0) {
        ws.n_tab[0] = ws.n_tab[1] = 0u;
    }
#pragma unroll 1
    for (int f = 0; f < A.n_frames; ++f) {
#if MBE_U_LOCKSTEP
        __syncthreads();
#endif
        if (!live) {
            continue;
        }
        const size_t idx = (size_t)(A.io_base + s) * A.n_frames + f;
        const uint32_t* d = A.desc + ((size_t)s * A.n_frames + f) * DESC_WORDS;
        const unsigned ia = tb & 3u;
        const bool hit = (tb & 4u) != 0u;
        tb = (ia == 0u) ? 2u : ia - 1u;
        const uint32_t* dw = d;   // frame f's words 0..7 and, at dw + dov, its overlap
        int dov = D_OV;
        if (A.noise_tab) {
            cp_async_wait_all();
            __syncwarp();
            if (f + 1 < A.n_frames && noise_prefetch(ws.dstage[(f + 1) & 1], A.noise_tab, bk, ws.buf[tb], lane)) {
                tb |= 4u;
            }
            dw = ws.dstage[f & 1];
            dov = 8;
        }
        float* Af = ws.buf[ia];
        float* Bf = ws.buf[ia == 2u ? 0u : ia + 1u];
        unsigned ops = dw[D_OPS];
        // the noise spectrum depends on the descriptor alone, not on the previousUw ops: it is ready before they run
        if (dw[D_INFO] & 1u) {
            for (int i = lane; i < 129; i += 32) {
                ws.scale[i] = 0.0f;
            }
            if (A.counters && lane == 0) {
                ++ws.n_tab[hit ? 0 : 1];
            }
            if (!hit) {
                split_noise(Af, __uint_as_float(dw[D_SEED]), dw + dov, bt, lane);
                __syncwarp();
                rfft256_forward_inl(Af, Bf, bt->tw, lane);
            } else {
                __syncwarp();
            }
        }
        if (A.noise_tab && f + 2 < A.n_frames) {
            __syncwarp();   // (every lane has read frame f's staged words)
            stage_desc(ws.dstage[f & 1], d + 2 * DESC_WORDS, lane);
        }
#pragma unroll 1
        while (ops) {
            const unsigned op = ops & 15u;
            ops >>= 4;
            if (op == OP_SYNTH) {
                const unsigned info = d[D_INFO];
                const int L = (int)((info >> 8) & 255u);
                float tail[4], voiced[5];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    tail[q] = __uint_as_float(h_enh[UW_WORD + 128 + 32 * q + lane]);
                }
#pragma unroll
                for (int q = 0; q < 5; ++q) {
                    voiced[q] = __uint_as_float(d[D_VOICED + 32 * q + lane]);
                }
                split_unvoiced_shape(ws, Af, Bf, d, L, __uint_as_float(d[D_CW0]), d[D_CU], d[D_CU + 1], bt, lane);
                const float* Ab = Af;
                const float inv = 1.0f / (float)NFFT;
#pragma unroll
                for (int cc = 0; cc < 5; ++cc) {
                    const int n = 32 * cc + lane;
                    const float den = bt->wola_den[n];
                    const float ps = (cc < 4) ? tail[cc < 4 ? cc : 0] : 0.0f;
                    const float cs = (n - 32 >= 0) ? (Ab[n - 32] * inv) : 0.0f;
                    float v = voiced[cc];
                    if (den > 1e-10f) {
                        v += ((bt->wola_wp[n] * ps) + (bt->wola_wc[n] * cs)) / den;
                    }
                    if (v > MBE_CLIP_F) {
                        v = MBE_CLIP_F;
                    } else if (v < -MBE_CLIP_F) {
                        v = -MBE_CLIP_F;
                    }
                    const size_t o = idx * NS + n;
                    if (A.pcmf) {
                        A.pcmf[o] = ref_nan(v * A.pcmf_scale);
                    }
                    if (A.pcm) {
                        A.pcm[o] = float_to_short(v);
                    }
                }
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const uint32_t v = __float_as_uint(Ab[32 * q + lane] * inv);
                    h_cur[UW_WORD + 32 * q + lane] = v;
                    h_enh[UW_WORD + 32 * q + lane] = v;
                }
                __syncwarp();
            } else if (op == OP_PREV_FROM_CUR) {
                uw_copy(h_prev, h_cur, lane);
            } else if (op == OP_CUR_FROM_PREV) {
                uw_copy(h_cur, h_prev, lane);
            } else if (op == OP_ENH_FROM_CUR) {
                uw_copy(h_enh, h_cur, lane);
            } else if (op == OP_CUR_FROM_ENH) {
                uw_copy(h_cur, h_enh, lane);
            } else if (op == OP_SPILL_FROM_CUR) {
                uw_copy(h_spill, h_cur, lane);
            } else if (op == OP_CUR_FROM_SPILL) {
                uw_copy(h_cur, h_spill, lane);
            } else if (op == OP_ZERO_CUR) {
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    h_cur[UW_WORD + 32 * q + lane] = 0u;
                }
            }
        }
    }
    cp_async_wait_all();
    if (A.counters && live && lane == 0) {
        atomicAdd(&A.counters[4], (unsigned long long)ws.n_tab[0]);
        atomicAdd(&A.counters[5], (unsigned long long)ws.n_tab[1]);
    }
}

}  // namespace mbe
