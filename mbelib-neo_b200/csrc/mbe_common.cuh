// Shared declarations for the B200 IMBE/AMBE decoder kernels: state layout, lookup tables that are
// filled on the host at context creation, per-warp shared-memory workspace.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/mbe_b200.h"

namespace mbe {

constexpr unsigned FULL = 0xffffffffu;
constexpr int NS = 160;     // samples per frame
constexpr int NFFT = 256;   // unvoiced FFT length
constexpr int WIN_PREV = 164;  // BlockTables::voiced_win: where the previous-frame half of the window starts
constexpr int MAXL = 56;    // max harmonics

// Device image of the reference's `struct mbe_parameters` (include/mbelib-neo/mbelib.h:88-137).
// Byte-identical layout: it is the import/export format of the C-ABI.
struct Parms {
    float w0;
    int L;
    int K;
    int Vl[57];
    float Ml[57];
    float log2Ml[57];
    float PHIl[57];
    float PSIl[57];
    float gamma;
    uint32_t tonePhase;
    int swn;
    float localEnergy;
    int amplitudeThreshold;
    float errorRate;
    int errorCountTotal;
    int errorCount4;
    int repeatCount;
    float mutingThreshold;
    float previousUw[256];
    float noiseSeed;
    float noiseOverlap[96];
};
static_assert(sizeof(Parms) == MBE_B200_PARMS_BYTES, "mbe_parms layout");

// The same struct without its two bulk arrays: what the kernel keeps in shared memory for prev_mp and
// prev_mp_enhanced (their previousUw / noiseOverlap stay in the stream's HBM slot and are only touched
// by whole-struct copies and by the overlap-add).  Words 0..297 are laid out exactly like Parms.
struct ParmsSmall {
    float w0;
    int L;
    int K;
    int Vl[57];
    float Ml[57];
    float log2Ml[57];
    float PHIl[57];
    float PSIl[57];
    float gamma;
    uint32_t tonePhase;
    int swn;
    float localEnergy;
    int amplitudeThreshold;
    float errorRate;
    int errorCountTotal;
    int errorCount4;
    int repeatCount;
    float mutingThreshold;
    float noiseSeed;
};
// prev_mp in shared memory: only what the decoders read every frame (prediction source, error-rate filter,
// repeat counters).  Its Vl / PHIl[1..56] / PSIl words stay in the stream's HBM image like the bulk arrays; they
// are only moved by whole-struct copies (repeat, erasure model).
struct PrevSmall {
    float w0;
    int L;
    int K;
    float Ml[57];
    float log2Ml[57];
    float PHIl0;                      // PHIl[0]: the reference's prediction reads log2Ml[57] == PHIl[0]
    float gamma;
    uint32_t tonePhase;
    int swn;
    float localEnergy;
    int amplitudeThreshold;
    float errorRate;
    int errorCountTotal;
    int errorCount4;
    int repeatCount;
    float mutingThreshold;
    float noiseSeed;
};
// prev_mp_enhanced in shared memory: the synthesis continuity state; its log2Ml stays in HBM.
struct EnhSmall {
    float w0;
    int L;
    int K;
    int Vl[57];
    float Ml[57];
    float PHIl[57];
    float PSIl[57];
    float gamma;
    uint32_t tonePhase;
    int swn;
    float localEnergy;
    int amplitudeThreshold;
    float errorRate;
    int errorCountTotal;
    int errorCount4;
    int repeatCount;
    float mutingThreshold;
    float noiseSeed;
};
constexpr int PREV_WORDS = 129, ENH_WORDS = 242;
static_assert(sizeof(PrevSmall) == PREV_WORDS * 4 && sizeof(EnhSmall) == ENH_WORDS * 4, "compact layouts");
// word j of the compact struct <-> word of the 651-word mbe_parms image
__host__ __device__ constexpr int prev_word(int j) { return j < 3 ? j : (j < 118 ? j + 57 : (j < 128 ? j + 170 : 554)); }
__host__ __device__ constexpr int enh_word(int j) { return j < 117 ? j : (j < 241 ? j + 57 : 554); }
static_assert(prev_word(3) == 60 && prev_word(117) == 174 && prev_word(118) == 288 && prev_word(127) == 297, "prev map");
static_assert(enh_word(116) == 116 && enh_word(117) == 174 && enh_word(231) == 288 && enh_word(240) == 297, "enh map");
// mbe_parms words of prev_mp that are NOT in PrevSmall: Vl[0..56] = 3..59, PHIl[1..56] + PSIl[0..56] = 175..287 (170 words);
// of prev_mp_enhanced: log2Ml[0..56] = 117..173 (57 words)
__host__ __device__ constexpr int prev_home_word(int j) { return j < 57 ? 3 + j : 118 + j; }
constexpr int PREV_HOME_WORDS = 170, ENH_HOME_WORD0 = 117, ENH_HOME_WORDS = 57;
static_assert(prev_home_word(56) == 59 && prev_home_word(57) == 175 && prev_home_word(169) == 287, "prev home map");

constexpr int HEAD_WORDS = 298;       // w0 .. mutingThreshold
constexpr int UW_WORD = 298;          // previousUw[256]
constexpr int SEED_WORD = 554;        // noiseSeed
constexpr int OVERLAP_WORD = 555;     // noiseOverlap[96]
static_assert(sizeof(ParmsSmall) == (HEAD_WORDS + 1) * 4, "ParmsSmall layout");
static_assert(offsetof(Parms, previousUw) == UW_WORD * 4 && offsetof(Parms, noiseSeed) == SEED_WORD * 4 &&
                  offsetof(Parms, noiseOverlap) == OVERLAP_WORD * 4 && offsetof(Parms, mutingThreshold) == 297 * 4,
              "mbe_parms offsets");
constexpr int PARMS_WORDS = sizeof(Parms) / 4;            // 651
// NaN bit patterns at the library's boundary.  Every NaN the reference can produce on its x86-64 target comes from an invalid
// operation (0/0 in the enhancement of an erasure model, 0 * inf, ...) and is the SSE default NaN 0xffc00000, which then
// propagates unchanged; the GPU's arithmetic produces (and propagates) its canonical NaN 0x7fffffff instead.  Both decode
// identically afterwards; only the bit pattern a caller sees differs, so float words that leave the library - exported
// mbe_parms images, float PCM - carry the reference's pattern.  (NaNs with other payloads, i.e. imported ones, are left alone.)
__host__ __device__ constexpr bool parms_word_is_float(int w) {
    return w == 0 || (w >= 60 && w <= 288) || w == 291 || w == 293 || w >= 297;
}
__device__ __forceinline__ uint32_t ref_nan_word(uint32_t v) { return v == 0x7fffffffu ? 0xffc00000u : v; }
__device__ __forceinline__ float ref_nan(float x) { return __uint_as_float(ref_nan_word(__float_as_uint(x))); }
__device__ __forceinline__ uint32_t ref_nan_parms_word(int w, uint32_t v) { return parms_word_is_float(w) ? ref_nan_word(v) : v; }
constexpr int RNG_WORDS = 4;                              // comfort lo, comfort hi, uv seed, uv override
constexpr int SPILL_WORD = 3 * PARMS_WORDS + RNG_WORDS;   // a fourth mbe_parms image: scratch of the AMBE+2 replay path
constexpr int STATE_WORDS = 4 * PARMS_WORDS + RNG_WORDS;  // per stream in HBM: cur, prev, enh, rng, scratch (10432 B)

// Tables computed on the host when a context is created (host libm = the reference's libm) and kept
// in HBM; hot ones are staged into shared memory per block.
// rows of DevTables::cosw
constexpr int COSW_IMBE = 0;                 // + b0 (0..207)
constexpr int COSW_A2450 = 208;              // + b0 (0..119)
constexpr int COSW_A2450_SILENCE = 328;
constexpr int COSW_A2400 = 329;              // + b0 (0..125)
constexpr int COSW_A2400_SILENCE = 455;
constexpr int COSW_IMBE_DEFAULT = 456;
constexpr int COSW_AMBE_DEFAULT = 457;
constexpr int COSW_ROWS = 458;

struct DevTables {
    // DCT cosines (src/imbe/imbe7200x4400.c:97-111, src/ambe/ambe3600x2450.c:60-74)
    float ri6[36];      // [m-1][i-1]
    float ri8[64];
    float blk[1785];    // packed [ji][j][k]: blk_off[ji] + (j-1)*ji + (k-1), ji = 1..17
    int blk_off[18];
    // FFTPACK twiddles for N=256 (src/external/pffft/pffft.c:1231-1262)
    float tw[256];
    // b0 -> model tables
    float imbe_w0[256];
    unsigned char imbe_L[256];   // 0 = invalid (b0 > 207 or L out of 9..56)
    unsigned char imbe_K[256];   // K as mbe_convertImbe7100to7200 computes it (no validity check)
    unsigned char imbe_Kv[256];  // K for valid b0
    float a2450_w0[120];
    float a2450_w0_silence;
    float a2450_f0_silence;
    float a2400_f0[126];
    float a2400_w0[126];
    float a2400_w0_silence;
    float imbe_default_w0;
    int imbe_default_L;
    float ambe_default_w0;
    float log2_int[57];          // log2f((float)L)
    float ambe_rconst;           // (float)(1/(2*sqrt(2)))
    // LCG jump-ahead tables: x_k = (A[k]*x_0 + C[k]) mod m
    unsigned short pnA[116], pnC[116];  // PN de-scrambler, mod 65536
    unsigned uvA[161], uvC[161];        // unvoiced noise, mod 53125
    unsigned uvBA[96], uvBC[96];        // LCG^(53125 - 96 + k) = LCG^(k - 96) (full period): a frame's natural overlap word k
    unsigned long long cnA[161], cnC[161];  // comfort noise, mod 2^48
    // ECC
    unsigned short golay_par_hi[64], golay_par_lo[64];
    unsigned golay_cw[4096];            // all codewords, index = 12 data bits
    unsigned short ham_cw[2][2048];     // all Hamming(15,11) codewords in the reference's enumeration order
    unsigned short ham_rows[2][4];
    unsigned short ham_flip[2][16];
    unsigned char ham_par_hi[2][32], ham_par_lo[2][64];  // compacted parity of codeword (d << 6) / d
    // windows
    float uvwin[256];                   // 211-pt trapezoid centred at 128
    float wola_wp[160], wola_wc[160], wola_den[160];
    float voiced_win[324];
    unsigned short golay_fix[2048];
    // cos(l * w0), l = 1..56, for every fundamental the decoders can produce, generated ON THE DEVICE at context
    // creation by the reference's own rotation recurrence (mbelib.c:412-424) so the values are the ones the
    // enhancement would compute frame by frame.  Row r belongs to the fundamental cosw_w0[r]; a frame whose w0 is not
    // bitwise equal to its row's runs the recurrence itself.
    // channel map of the bit-packed input (mbe_b200_set_channel_map): frame position r*cols + c takes transmitted bit
    // chan_src[codec][pos] of the packed frame (0xffff: the position is not transmitted and reads 0); identity by default
    unsigned short chan_src[4][184];
    float cosw_w0[COSW_ROWS];
    float cosw[COSW_ROWS][57];
    // (sin, cos) of l * w0 as the kernel's sincosf port gives them (the oscillator step of harmonic l, mbelib.c:978-1011),
    // generated on the device; same row key and same bitwise row check as cosw
    float2 stepsc[COSW_ROWS][57];
};

// mode of the stream kernel
enum { MODE_FRAMES = 0, MODE_DATA = 1, MODE_SYNTH = 2 };

struct LaunchArgs {
    int codec, soft, mode;
    int first_stream, n_streams, n_frames;
    const uint8_t* frames;      // MODE_FRAMES: channel frames; MODE_DATA: parameter bits
    int16_t* pcm;
    float* pcmf;
    mbe_b200_result* results;
    uint8_t* bits;
    uint32_t* state;            // [max_streams][STATE_WORDS]
    const DevTables* tab;
    // MODE_SYNTH: cur/prev parameter blobs in device memory, [n][651] words each, updated in place
    uint32_t* synth_cur;
    uint32_t* synth_prev;
    const uint32_t* synth_seeds;
    uint32_t* synth_rng;        // MODE_SYNTH: [n][4] RNG words in/out (overrides synth_seeds)
    unsigned long long* dbg;    // MBE_STAGE_TIMING builds: 16 accumulated per-stage cycle counters
    int packed_bytes;           // bit-packed input: bytes per frame (transmitted bits of the channel map, rounded up)
    float pcmf_scale;           // float PCM is multiplied by this on store: 1 (reference scale) or 7/32768 (normalised)
    uint32_t* desc;             // split path: frame descriptors [n_streams][n_frames][DESC_WORDS] (mbe_split.cuh)
    int io_base;                // stream s of the launch is element io_base + s of the caller's frame / PCM / result arrays
    // indexed calls (mbe_b200_process_indexed*): element e = slot_base + io_base + s of the call decodes stream slot
    // slots[e] (slots == nullptr: the contiguous range first_stream + s).  The element owns its slot only when the slot is in
    // [0, max_streams) and claim[slot] holds its own tag (claim_tag: the first occurrence of a repeated slot wins).
    const int32_t* slots;
    const unsigned long long* claim;
    unsigned epoch;
    int slot_base, max_streams;
};

// the claim an element of an indexed call leaves on its slot: later calls have larger epochs, earlier elements larger tags
__host__ __device__ __forceinline__ unsigned long long claim_tag(unsigned epoch, int e) {
    return ((unsigned long long)epoch << 32) | (0xffffffffu - (unsigned)e);
}

// state slot of stream s of a launch (LaunchArgs, SynthArgs): the contiguous range, or the slot an indexed call lists
template <class Args>
__device__ __forceinline__ int slot_of(const Args& A, int s) {
    return A.slots ? A.slots[A.slot_base + A.io_base + s] : A.first_stream + s;
}


// Tables every warp of a block reads with lane-varying indices on the synthesis path, staged into
// shared memory once per block (5.3 KB).
struct __align__(16) BlockTables {
    // 321-pt voiced window Ws (mbelib_const.h) as its two halves: a current-frame component is weighted by Ws[n], a
    // previous-frame one by Ws[160 + n], n = 0..159.  The halves sit 164 floats apart: the lanes of a warp broadcast-load
    // (LDS.128) from both at the same n, and 160 floats apart they would hit the same four banks (59 % of the kernel's
    // excess shared-memory wavefronts in profiles/r01z_imbe_hard_kernel_ncu_details.txt)
    float voiced_win[328];   // [0, 160): Ws[n];  [164, 324): Ws[160 + n]
    float tw[256];           // FFTPACK twiddles
    float uvwin[256];        // unvoiced analysis window, centred at 128
    float wola_wp[160], wola_wc[160], wola_den[160];
    uint2 uv_jump[32];       // unvoiced-noise LCG jump-ahead by `lane` steps: x -> (x * .x + .y) mod 53125
};

// Streams (= warps) per block.  The block walks its streams' frames in lockstep: per frame every warp
// decodes its own stream, then the block pools the oscillator components of all its streams and
// spreads them evenly over all lanes (voiced_bank_block), then every warp finishes its own stream.
#ifndef MBE_WPB
#define MBE_WPB 14
#endif
#ifndef MBE_MINB
#define MBE_MINB 2
#endif
constexpr int WARPS_PER_BLOCK = MBE_WPB;
constexpr int MIN_BLOCKS_PER_SM = MBE_MINB;

// The reference's thread-local RNG state, per stream (mbe_adaptive.c:29-30, mbe_unvoiced_fft.c:29-30)
struct StreamRng {
    unsigned long long comfort;  // 48-bit comfort-noise LCG state
    unsigned uv_seed;            // unvoiced cold-start seed override
    unsigned uv_override;        // consumed by the first cold start
};

// Per-warp shared-memory workspace: one warp owns one stream for the whole launch.
struct __align__(16) WarpWS {
    StreamRng rng;
    float out[NS];                        // the frame's 160 float samples (lane i owns i, 32+i, ...)
    // The three mbe_parms of the stream WITHOUT their bulk arrays (previousUw / noiseOverlap stay in the
    // stream's HBM slot); 16-byte aligned for 128-bit struct copies.
    ParmsSmall cur;
    short w0row;                          // DevTables::cosw row of the fundamental this frame's decoder chose (unverified)
    short w0row_prev;                     // row that matched the previous enhanced frame
    short w0row_enh;                      // candidate row of prev_mp_enhanced's fundamental (checked bitwise at use)
    short pad0;
    // split path (mbe_split.cuh): the previousUw copies this frame's state machine asked for, 4 bits each, in order
    unsigned ops, nops, pad1, pad2;
    PrevSmall prev;
    EnhSmall enh;
    int ncomp;                            // oscillator components of this frame (0: no voiced synthesis)
    unsigned k2mask;                      // list positions (< 32) of phase-interpolated harmonics
    unsigned short off[WARPS_PER_BLOCK + 3];  // this warp's copy of the block's slot offsets (prefix of padded counts)
    // interpolated harmonics of the block this warp renders in this round (indices into the block's list): up to 3 as a warp
    // without an oscillator pass plus up to 7 dealt round-robin (7 per stream at most, W streams over W warps), so 10
    unsigned short interp_item[10];
    unsigned char comp[112];              // component descriptor: harmonic << 2 | kind
    // LAST member: the parameter kernel of the multi-kernel path with hard-decision input only needs the decode scratch
    // (WS_STRIDE_SMALL), so its per-warp stride stops short of the tile
    union __align__(16) {
        float tile[32 * 32];              // voiced bank: [sample][slot] pre-weighted contributions, XOR-swizzled (tile_at)
        struct {
            float a[324];                 // FFT ping buffer (windowed noise on entry); 324: padded pass layouts
            float b[324];                 // FFT pong buffer
            float scale[132];             // per-bin unvoiced band scale
        } fft;
        struct {                          // front-end / parameter decode scratch (dead before synthesis starts)
            float tmp[128];               // per-harmonic terms [1..56], DCT coefficients [64+l]
            float Tl[60];
            int field[58];                // IMBE quantiser words b1..bL+1
            unsigned rowbits[8];
            unsigned char rel[8 * 24];    // soft-bit reliabilities of the frame
        } dec;
        float nz[57];                     // white-noise samples 1..56 of the frame (phase randomisation; dead before the bank)
    } u;                                  // 16-byte aligned: rows are read with LDS.128
};
static_assert(sizeof(((WarpWS*)0)->u) >= 4096 && sizeof(((WarpWS*)0)->out) >= 608, "soft-decision scratch (SoftScratch)");
static_assert(offsetof(WarpWS, u) % 16 == 0 && sizeof(WarpWS) % 16 == 0 && sizeof(BlockTables) % 16 == 0 &&
                  offsetof(WarpWS, cur) % 16 == 0,
              "LDS.128 alignment");
// per-warp stride of the multi-kernel path's parameter kernel on hard-decision input: everything up to the union + the
// decode scratch / the 176-float scratch of the spectral enhancement (no tile, no transforms in that kernel)
constexpr size_t WS_DEC_BYTES = (sizeof(((WarpWS*)0)->u.dec) + 15) & ~(size_t)15;
static_assert(WS_DEC_BYTES >= 176 * 4 + 16, "spectral_enhance scratch");
constexpr size_t WS_STRIDE_SMALL = offsetof(WarpWS, u) + WS_DEC_BYTES;
#ifndef MBE_PWPB
#define MBE_PWPB 18
#endif
#ifndef MBE_PMINB
#define MBE_PMINB 2
#endif
constexpr int P_WARPS = MBE_PWPB;   // warps per block of that kernel (56 registers per thread at two blocks of 18 warps per SM)
constexpr int P_MINB = MBE_PMINB;

struct BlockShared {
    int cnt[2][WARPS_PER_BLOCK + 2];      // per stream: component count of the current frame (double-buffered by frame parity)
    int n_interp[2];                      // phase-interpolated harmonics of the block's streams in this frame
    unsigned short interp[2][WARPS_PER_BLOCK * 7 + 2];  // owner stream << 8 | list position (at most 7 per stream: l < 8)
    float interp_a1[2][WARPS_PER_BLOCK * 7 + 2];        // per item: the phase increment per sample, pw0*l + delta-omega
};

// MBE_STAGE_TIMING=1 builds accumulate per-stage clock64() deltas per warp into LaunchArgs.dbg (profiling aid)
#ifndef MBE_STAGE_TIMING
#define MBE_STAGE_TIMING 0
#endif
#if MBE_STAGE_TIMING
struct StageTimer {
    long long acc[16];
    long long last;
};
#define STAGE_T(i) do { const long long _t = clock64(); tm.acc[i] += _t - tm.last; tm.last = _t; } while (0)
#else
struct StageTimer {};
#define STAGE_T(i) do { } while (0)
#endif

}  // namespace mbe
