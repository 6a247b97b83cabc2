/*
 * TEST INFRASTRUCTURE - CPU oracle for the batched IMBE/AMBE decode+synthesis hot path.
 *
 * Plain-C restatement of the algorithm the reference (arancormonk/mbelib-neo v2.0.0) runs between
 * "frame bits in" and "int16 PCM out".  Only tests/, __graft_entry__.smoke() and bench.py's
 * cpu_baseline / --impl reference legs may load this library; the product (libmbe_b200.so) never
 * links or calls it.
 *
 * Parity status: PINNED.  tests/test_oracle_vs_ref.py checks it bit-for-bit against the compiled,
 * unmodified reference (oracle/_ref/libmberef.so, built by oracle/Makefile from /root/reference) on
 * seeded inputs for all four codecs, hard and soft, and tests/test_oracle_kat.py checks the golden
 * vectors the reference's own tests hold (tests/test_golden_pcm.c:78-84, tests/test_ecc.c, ...).
 *
 * The reference's thread-local hidden state (comfort-noise LCG48, unvoiced cold-start seed override;
 * src/core/mbe_adaptive.c:29-30, src/core/mbe_unvoiced_fft.c:29-30) is an explicit per-stream
 * `mbo_rng` here, exactly as the device keeps it.
 */
#ifndef MBE_ORACLE_H
#define MBE_ORACLE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Same layout as the reference's `struct mbe_parameters` (include/mbelib-neo/mbelib.h:88-137):
 * it is the import/export format of the drop-in boundary. sizeof == 2604. */
typedef struct mbo_parms {
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
} mbo_parms;

typedef struct mbo_soft_bit {
    uint8_t bit;
    uint8_t reliability;
} mbo_soft_bit;

typedef struct mbo_result {
    int c0_errors;
    int protected_errors;
    int c4_errors;
    int total_errors;
    unsigned flags;
} mbo_result;

/* Per-stream replacement for the reference's thread-locals. */
typedef struct mbo_rng {
    uint64_t comfort_seed48; /* java.util.Random style 48-bit LCG state */
    uint32_t uv_seed;        /* unvoiced LCG cold-start seed override */
    int uv_override;         /* consumed by the first cold start */
} mbo_rng;

enum { MBO_IMBE7200 = 0, MBO_IMBE7100 = 1, MBO_AMBE2400 = 2, MBO_AMBE2450 = 3 };

#define MBO_FLAG_SOFT_INPUT 0x0001u
#define MBO_FLAG_C0_VALID   0x0002u
#define MBO_FLAG_C4_VALID   0x0004u
#define MBO_FLAG_TONE       0x0010u
#define MBO_FLAG_ERASURE    0x0020u
#define MBO_FLAG_REPEAT     0x0040u
#define MBO_FLAG_MUTE       0x0080u
#define MBO_ERR_ARGUMENT    (-1)
#define MBO_ERR_BITS        (-2)

/* geometry */
int mbo_frame_bits(int codec);  /* 184 / 168 / 96 / 96 */
int mbo_param_bits(int codec);  /* 88 / 88 / 49 / 49 */

/* RNG + state */
void mbo_rng_default(mbo_rng* rng);                /* fresh-thread state */
void mbo_rng_seed(mbo_rng* rng, uint32_t seed);    /* == mbe_setThreadRngSeed */
void mbo_init_parms(mbo_parms* cur, mbo_parms* prev, mbo_parms* enh); /* == mbe_initMbeParms */

/* ECC primitives (src/ecc/ecc.c) */
int mbo_check_golay_block(long* block);
int mbo_golay2312(const char* in, char* out);
int mbo_golay2312_soft(const mbo_soft_bit* in, char* out);
int mbo_hamming1511(const char* in, char* out, int variant7100);
int mbo_hamming1511_soft(const mbo_soft_bit* in, char* out, int variant7100);
void mbo_ecc_blocks(int code, int soft, int fast, int n, const uint8_t* in, uint8_t* out, int32_t* status, int n_threads);

/* frame bits -> parameter bits (mbe_decode<Codec>[Soft]Frame) */
int mbo_decode_frame(int codec, int soft, const void* frame, char* bits, mbo_result* result);

/* parameter bits -> model parameters (mbe_decode*Parms) */
int mbo_decode_imbe4400_parms(const char* d, mbo_parms* cur, mbo_parms* prev);
int mbo_decode_ambe2400_parms(const char* d, mbo_parms* cur, mbo_parms* prev);
int mbo_decode_ambe2450_parms(const char* d, mbo_parms* cur, mbo_parms* prev, int total_errors);

/* synthesis building blocks (src/core) */
float mbo_spectral_amp_enhance(mbo_parms* cur);                              /* returns pre-enhancement Rm0 */
void mbo_adaptive_smoothing(mbo_parms* cur, const mbo_parms* prev, int has_rm0, float rm0);
void mbo_synthesize_speech(float* out, mbo_parms* cur, mbo_parms* prev, int has_rm0, float rm0, mbo_rng* rng);
void mbo_comfort_noise(float* out, mbo_rng* rng);
void mbo_synthesize_tone(float* out, const char* ambe_d, mbo_parms* cur);
void mbo_synthesize_tone_dstar(float* out, mbo_parms* cur, int id1);
void mbo_float_to_short(const float* in, short* out);
void mbo_noise_with_overlap(float* buf256, float* seed, float* overlap96, mbo_rng* rng);
void mbo_fft256_forward_ordered(const float* in, float* out);
void mbo_fft256_backward_ordered(const float* in, float* out);

/* parameter bits -> float PCM (mbe_process<Codec>Dataf) and frame -> float PCM (mbe_process<Codec>[Soft]Framef) */
int mbo_process_data(int codec, float* out, mbo_result* result, const char* bits, mbo_parms* cur, mbo_parms* prev,
                     mbo_parms* enh, mbo_rng* rng);
int mbo_process_frame(int codec, int soft, float* out, mbo_result* result, const void* frame, char* bits,
                      mbo_parms* cur, mbo_parms* prev, mbo_parms* enh, mbo_rng* rng);

/* Batch driver with the same signature as oracle/ref_bench.c:ref_bench_run (single thread per call
 * unless n_threads > 1; streams are independent). Returns seconds. */
double mbo_run(int codec, int soft, int n_streams, int n_frames, const uint8_t* frames, const uint32_t* seeds,
               int16_t* pcm, float* pcmf, int32_t* results, uint8_t* bits, void* state, int n_threads);

/* mbo_run that also reports every frame's oscillator-bank work, work[stream][frame][3] (may be null):
 *   [0] oscillator slots: one per interpolated harmonic (l < 8, voiced in both frames, |cur w0 - prev w0| < 0.1 cur w0),
 *       one per other windowed component of the previous and of the current frame whose gain 2 Ml is not exactly 0 or
 *       whose phase is not finite (the device's build_components rule);
 *   [1] of them interpolated harmonics;
 *   [2] 1 when the frame runs the speech synthesis (0 for tone, silence, comfort-noise and rejected frames).
 * Everything else it returns is what mbo_run returns. */
double mbo_run_work(int codec, int soft, int n_streams, int n_frames, const uint8_t* frames, const uint32_t* seeds,
                    int16_t* pcm, float* pcmf, int32_t* results, uint8_t* bits, void* state, int32_t* work,
                    int n_threads);

#ifdef __cplusplus
}
#endif
#endif
