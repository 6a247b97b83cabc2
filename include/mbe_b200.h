/*
 * mbe_b200.h - C-ABI of the B200-native batched IMBE/AMBE decoder (libmbe_b200.so).
 *
 * Drop-in boundary for the decode-and-synthesis hot path of arancormonk/mbelib-neo v2.0.0.  Every entry
 * point is the batched form of one family of calls in the reference's public header
 * (/root/reference/include/mbelib-neo/mbelib.h, cited per function below): element [s][f] of a batch has
 * exactly the per-call semantics of the reference function applied to stream s's state, frames in order.
 *
 * Conventions
 *   - plain C, no CUDA/torch types: device pointers are `void*`/typed pointers into device memory,
 *     CUDA streams are passed as `void*` (a cudaStream_t; NULL = the context's own stream).
 *   - codec ids: MBE_B200_IMBE7200X4400 (P25 Phase 1, char[8][23]), MBE_B200_IMBE7100X4400
 *     (ProVoice, char[7][24]), MBE_B200_AMBE3600X2400 (D-STAR, char[4][24]),
 *     MBE_B200_AMBE3600X2450 (DMR/NXDN AMBE+2, char[4][24]).
 *   - hard frames: one byte per bit (0/1), laid out [stream][frame][rows*cols] exactly like the
 *     reference's `char fr[R][C]`; soft frames: `mbe_soft_bit` pairs {bit, reliability}
 *     (mbelib.h:148-151), i.e. 2 bytes per bit, same order.
 *   - PCM: int16 [stream][frame][160] (8 kHz, 20 ms) and/or float [stream][frame][160] in the
 *     reference's float scale (mbelib.h:16-20).
 *   - per-frame status: `mbe_b200_result` = the reference's mbe_process_result (mbelib.h:180-191) plus
 *     the call's return value (`status`: >= 0 total corrected errors, MBE_STATUS_INVALID_ARGUMENT (-1),
 *     MBE_STATUS_INVALID_BITS (-2)).  A frame with negative status leaves the stream state untouched
 *     and produces silence; its parameter-bit output (`bits`) reads all zero and, on the process_data
 *     path, its result element is the caller's input with only `.status` replaced (the reference
 *     returns before touching either; a batched output array has no "untouched" - check `.status`).
 *   - per-stream state lives on the device: the reference's caller-owned triplet cur_mp / prev_mp /
 *     prev_mp_enhanced (3 x 2604 bytes, `struct mbe_parameters` layout, mbelib.h:88-137) plus the
 *     reference's thread-local RNG state (comfort-noise LCG48 and unvoiced cold-start seed,
 *     src/core/mbe_adaptive.c:29-30, src/core/mbe_unvoiced_fft.c:29-30) made per-stream.
 *   - every function returns 0 on success or a negative MBE_B200_E_* code; mbe_b200_last_error()
 *     gives the text.  There is NO CPU fallback: without a CUDA device create() fails.
 */
#ifndef MBE_B200_H
#define MBE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MBE_B200_API __attribute__((visibility("default")))

enum {
    MBE_B200_IMBE7200X4400 = 0,
    MBE_B200_IMBE7100X4400 = 1,
    MBE_B200_AMBE3600X2400 = 2,
    MBE_B200_AMBE3600X2450 = 3
};

#define MBE_B200_SAMPLES_PER_FRAME 160
#define MBE_B200_PARMS_BYTES       2604 /* sizeof(mbe_parms) */

/* call-level error codes */
#define MBE_B200_E_ARG    (-1) /* bad argument (NULL pointer, range, codec id) */
#define MBE_B200_E_CUDA   (-2) /* CUDA runtime error, see mbe_b200_last_error() */
#define MBE_B200_E_NOGPU  (-3) /* no usable CUDA device - the product has no CPU path */

/* per-frame result: return value + mbe_process_result (mbelib.h:180-191; flags mbelib.h:153-166) */
typedef struct mbe_b200_result {
    int32_t status;           /* what the reference call would have returned */
    int32_t c0_errors;
    int32_t protected_errors;
    int32_t c4_errors;
    int32_t total_errors;
    uint32_t flags;           /* MBE_PROCESS_FLAG_* bit values of the reference */
} mbe_b200_result;

typedef struct mbe_b200_ctx mbe_b200_ctx;

/* ---- context: owns device tables, the per-stream state pool and staging buffers ---------------- */
MBE_B200_API int mbe_b200_create(mbe_b200_ctx** out, int device_ordinal, int max_streams);
MBE_B200_API void mbe_b200_destroy(mbe_b200_ctx* ctx);
MBE_B200_API const char* mbe_b200_last_error(const mbe_b200_ctx* ctx); /* ctx may be NULL: last create() error */
MBE_B200_API const char* mbe_b200_version(void);
MBE_B200_API int mbe_b200_geometry(int codec, int* frame_bits, int* param_bits); /* 184/168/96/96, 88/88/49/49 */
MBE_B200_API int mbe_b200_device_count(void); /* usable CUDA devices (0 when there is none or the driver is missing) */
/* Pinned (page-locked) host memory.  The reference's contract is "the caller owns every buffer" (mbelib.h:28-30); the
 * host-pointer entry points below accept any host pointer, but only page-locked buffers move at full link speed and overlap
 * with the kernels (a pageable 1 GB PCM buffer costs 3x on one GPU).  A plain-C caller that does not link the CUDA runtime
 * allocates its frame / PCM / result arrays here, or registers arrays it already owns.  Portable: valid for every device
 * of the process (mbe_b200_pool_*).  No context needed; errors: mbe_b200_last_error(NULL). */
MBE_B200_API int mbe_b200_host_alloc(void** out, size_t bytes);
MBE_B200_API int mbe_b200_host_free(void* p);
MBE_B200_API int mbe_b200_host_register(void* p, size_t bytes);
MBE_B200_API int mbe_b200_host_unregister(void* p);
/* kernel launches issued by this context so far (bench.py reports it as gpu_launches) */
MBE_B200_API long long mbe_b200_launch_count(const mbe_b200_ctx* ctx);
/* One stream, one frame, caller-owned state - the reference's call shape (mbe_process<Codec>[Soft]Frame[f] / Data[f]) in one
 * call: the {cur_mp, prev_mp, prev_mp_enhanced} triplet (3 x 2604 bytes) and the calling thread's four RNG words go to stream
 * slot `stream`, ONE frame is decoded and synthesised, both come back - one upload, one download, one synchronisation.
 * kind: 0 hard channel frame, 1 soft channel frame (mbe_soft_bit pairs), 2 parameter bits (`result` is then the IN/OUT decode
 * context of mbe_process<Codec>Data).  result->status < 0 (invalid bits / argument): nothing else is written, like the
 * reference's early return.  At least one of pcm / pcmf; bits may be NULL.  This is what the single-stream shim is built on;
 * throughput callers use the batched entry points. */
MBE_B200_API int mbe_b200_single_frame(mbe_b200_ctx* ctx, int codec, int kind, int stream, const void* frame,
                                       void* parms_triplet, uint32_t* rng_words4, int16_t* pcm, float* pcmf,
                                       mbe_b200_result* result, uint8_t* bits);
/* Kernel path of the frame entry points (process_frames*, process_data*): 0 = one fused kernel per batch, 1 = a parameter
 * kernel (ECC, decode, state machine, enhancement) that leaves a descriptor per frame + a synthesis kernel (oscillator
 * bank, FFT / overlap-add, PCM: a bank kernel and an unvoiced kernel) - DESIGN 4.5.  Results are bit-identical; the
 * default is 1 (MBE_B200_SPLIT in the environment overrides it).  kernel_path() returns the current setting. */
MBE_B200_API int mbe_b200_set_kernel_path(mbe_b200_ctx* ctx, int path);
MBE_B200_API int mbe_b200_kernel_path(const mbe_b200_ctx* ctx);
/* Measurement aid (bench.py): while enabled, every launch of the frame kernels is bracketed by a CUDA event pair on the
 * stream it runs on.  kernel_timing() synchronises and returns, per kernel kind (0 parameter or fused kernel, 1 bank
 * kernel, 2 unvoiced kernel), the summed device time in ms and the launch count since timing was enabled, plus the bank
 * kernel's work counters: [0] oscillator slots run (160 samples each), [1] of them phase-interpolated harmonics,
 * [2] frames synthesised, [3] 32-slot passes the bank kernel ran (slots / (32 x passes) = its lane fill).  The fused
 * kernel counts nothing. */
MBE_B200_API int mbe_b200_set_kernel_timing(mbe_b200_ctx* ctx, int enable);
MBE_B200_API int mbe_b200_kernel_timing(mbe_b200_ctx* ctx, double ms[3], long long launches[3], unsigned long long counters[4]);
/* The unvoiced kernel's counters over the same timing session: [0] frames whose noise spectrum came from the context's
 * noise table, [1] frames that computed their own (cold starts, imported states, MBE_B200_NOISE_TABLE=0).  Synchronises. */
MBE_B200_API int mbe_b200_noise_table_counters(mbe_b200_ctx* ctx, unsigned long long counters[2]);

/* ---- stream state ---------------------------------------------------------------------------
 * init_streams == per stream: mbe_setThreadRngSeed(seed) (mbelib.h:596; seeds==NULL: fresh-thread
 * default RNG state) followed by mbe_initMbeParms (mbelib.h:615).
 * export/import move [count][3] mbe_parms blobs {cur_mp, prev_mp, prev_mp_enhanced} to/from host
 * memory byte-for-byte; export_rng/import_rng move the per-stream RNG words
 * {comfort_seed48 lo, hi, unvoiced seed, override flag}. */
MBE_B200_API int mbe_b200_init_streams(mbe_b200_ctx* ctx, int first_stream, int count, const uint32_t* seeds);
MBE_B200_API int mbe_b200_export_state(mbe_b200_ctx* ctx, int first_stream, int count, void* parms_triplets);
MBE_B200_API int mbe_b200_import_state(mbe_b200_ctx* ctx, int first_stream, int count, const void* parms_triplets);
MBE_B200_API int mbe_b200_export_rng(mbe_b200_ctx* ctx, int first_stream, int count, uint32_t* rng_words4);
MBE_B200_API int mbe_b200_import_rng(mbe_b200_ctx* ctx, int first_stream, int count, const uint32_t* rng_words4);

/* ---- the hot path: frames -> PCM ---------------------------------------------------------------
 * Batched mbe_process<Codec>Frame / Framef / SoftFrame / SoftFramef
 * (mbelib.h:352-373, 429-447, 505-523, 564-582).  Streams first_stream .. first_stream+n_streams-1 each
 * consume n_frames consecutive frames.  Any of pcm / pcmf / results / bits may be NULL.
 *   _dev : all pointers are device pointers; the launch is asynchronous on `cuda_stream` (a cudaStream_t).  NULL selects
 *          the context's own stream, which is created cudaStreamNonBlocking: it does NOT synchronise with the legacy
 *          default stream, so order the producer of the inputs before the call (event / synchronize) or pass the
 *          producer's stream.
 *   host : pointers are host memory (pinned or pageable); H2D copy, kernel and D2H copy run on the
 *          context's stream and the call returns when the results are in host memory. */
MBE_B200_API int mbe_b200_process_frames_dev(mbe_b200_ctx* ctx, int codec, int soft, int first_stream, int n_streams,
                                             int n_frames, const uint8_t* d_frames, int16_t* d_pcm, float* d_pcmf,
                                             mbe_b200_result* d_results, uint8_t* d_bits, void* cuda_stream);
MBE_B200_API int mbe_b200_process_frames(mbe_b200_ctx* ctx, int codec, int soft, int first_stream, int n_streams,
                                         int n_frames, const uint8_t* frames, int16_t* pcm, float* pcmf,
                                         mbe_b200_result* results, uint8_t* bits);

/* The host-pointer call in two halves, for a server thread that has other work while a batch is in flight (filling the
 * next frame's buffer, driving the contexts of several GPUs from one thread): submit_frames queues copy-in, kernels and
 * copy-out and returns; the host buffers must stay valid and untouched until mbe_b200_wait() returns (use pinned memory,
 * pageable memory makes the copies synchronous).  One submission may be pending per context; every other call on the
 * context must wait for it first. */
MBE_B200_API int mbe_b200_submit_frames(mbe_b200_ctx* ctx, int codec, int soft, int first_stream, int n_streams,
                                        int n_frames, const uint8_t* frames, int16_t* pcm, float* pcmf,
                                        mbe_b200_result* results, uint8_t* bits);
MBE_B200_API int mbe_b200_wait(mbe_b200_ctx* ctx);
/* Float PCM scale (SURVEY 8(f)-3).  By default every `pcmf` output is in the reference's historical float scale
 * (roughly int16/7, what mbe_process<Codec>Framef returns).  With enable != 0 the samples are multiplied by
 * (7.0f / 32768.0f) on store, the normalisation include/mbelib-neo/mbelib.h:16-20 documents (about [-0.95, +0.95]
 * after the soft clip).  int16 outputs are not affected. */
MBE_B200_API int mbe_b200_set_normalized_float(mbe_b200_ctx* ctx, int enable);

/* Bit-packed channel frames (SURVEY 8(f)-1): the same hard-decision frames with eight channel bits per byte instead of
 * the reference's one `char` per bit (README.md:171-178 of the reference).  Bit k = r*cols + c of `fr[r][c]` is bit
 * 7 - (k & 7) of byte k >> 3 (MSB first); a frame takes mbe_b200_packed_frame_bytes(codec) = 23 / 21 / 12 / 12 bytes.
 * Semantics per frame are those of mbe_process<Codec>Frame[f]; a packed bit can only be 0 or 1, so
 * MBE_STATUS_INVALID_BITS cannot occur. */
MBE_B200_API int mbe_b200_packed_frame_bytes(int codec);
/* How a host-pointer call of n_streams streams is cut into pipeline chunks (host logic only, no device needed): writes
 * up to `cap` chunk sizes in stream order and returns the number of chunks (0 for an empty call).  Small batches are one
 * chunk; large ones are about 32 chunks of whole blocks-per-SM multiples, with pieces that double from / halve towards
 * the two ends so that the copy-in ahead of the first kernel and the copy-out behind the last one stay small.
 * MBE_B200_CHUNKS / MBE_B200_TAPER / MBE_B200_KSTREAMS (environment) override chunk count, smallest piece in blocks
 * (0 = no taper) and the number of compute streams; they are tuning knobs, results do not depend on them.  (On the
 * multi-kernel path a context rounds the body chunks of very large batches - a chunk of at least one full stream range -
 * to whole stream ranges; the plan reported here is the context-free one.) */
MBE_B200_API int mbe_b200_pipeline_plan(int n_streams, int* sizes, int cap);
/* Channel map (SURVEY 8(f)-1, on-device de-interleave): by default packed bit k is frame position k.  With a map,
 * the packed frame holds the n_bits transmitted bits of the air interface in transmission order (MSB first, n_bits <=
 * rows*cols, mbe_b200_channel_frame_bytes() bytes per frame) and transmitted bit k lands at frame position
 * map[k] = r*cols + c of the reference's `fr[r][c]`; positions no transmitted bit maps to read 0 (the unused corners of
 * the reference's bit planes).  The de-interleave schedule itself is the air interface's (P25 LDU, DMR burst, D-STAR,
 * ...) and is supplied by the caller; the reference leaves it to the caller too.  map == NULL restores the identity.
 * A configuration call: it synchronises the device.  Applies to mbe_b200_process_frames_packed[_dev] of that codec. */
MBE_B200_API int mbe_b200_set_channel_map(mbe_b200_ctx* ctx, int codec, const uint16_t* map, int n_bits);
MBE_B200_API int mbe_b200_channel_frame_bytes(const mbe_b200_ctx* ctx, int codec);
MBE_B200_API int mbe_b200_process_frames_packed_dev(mbe_b200_ctx* ctx, int codec, int first_stream, int n_streams,
                                                    int n_frames, const uint8_t* d_packed, int16_t* d_pcm, float* d_pcmf,
                                                    mbe_b200_result* d_results, uint8_t* d_bits, void* cuda_stream);
MBE_B200_API int mbe_b200_process_frames_packed(mbe_b200_ctx* ctx, int codec, int first_stream, int n_streams,
                                                int n_frames, const uint8_t* packed, int16_t* pcm, float* pcmf,
                                                mbe_b200_result* results, uint8_t* bits);

/* ---- indexed batches: any set of stream slots in one call -----------------------------------------------------
 * A server that gives each call a state slot when the call starts and frees it when the call ends has, at every 20 ms tick,
 * frames for a scattered subset of its slots.  An indexed call decodes that subset in one call: element i of the batch is
 * stream slot slots[i] (any order), and frames / PCM / float PCM / results / bits are laid out [i][frame][...] exactly like
 * stream i of a contiguous call; every element consumes n_frames frames with the semantics of the frame calls above.
 * `input` says what `in` holds (MBE_B200_INPUT_*; PACKED uses the codec's channel map, mbe_b200_set_channel_map).
 *   _dev    : d_slots and every buffer are device pointers, asynchronous on cuda_stream (as process_frames_dev).
 *   host    : slots and every buffer are host pointers (as process_frames); submit_indexed is its asynchronous half,
 *             completed by mbe_b200_wait (as submit_frames; the slot list must stay valid until then too).
 * Rejection: an element whose slot is outside [0, max_streams), or repeats a slot an earlier element of the same list
 * names, is rejected - all its frames read status MBE_STATUS_INVALID_ARGUMENT (-1) with every other result field zero,
 * zero PCM / float PCM / bits, and no stream state is touched (the indexed parameter-bit calls, whose results are
 * IN/OUT, echo the caller's result instead: mbe_b200_process_data_indexed).  Every other element decodes normally, so the first
 * occurrence of a repeated slot wins.  The check covers the whole list, on the device (_dev) as on the host calls.
 * The state calls below validate on the host instead: an out-of-range or repeated slot fails the whole call with
 * MBE_B200_E_ARG and nothing is touched.  n == 0 or n_frames == 0 returns 0 and launches nothing.
 * Concurrent calls (on different CUDA streams) whose slot sets overlap are the caller's error, as overlapping stream ranges
 * are for the contiguous calls.  Slot allocation stays with the caller. */
#define MBE_B200_INPUT_HARD   0 /* one byte per bit, fr[R][C] order */
#define MBE_B200_INPUT_SOFT   1 /* mbe_soft_bit pairs */
#define MBE_B200_INPUT_PACKED 2 /* 8 hard bits per byte; the codec's channel map applies */
MBE_B200_API int mbe_b200_process_indexed_dev(mbe_b200_ctx* ctx, int codec, int input, const int32_t* d_slots, int n,
                                              int n_frames, const uint8_t* d_in, int16_t* d_pcm, float* d_pcmf,
                                              mbe_b200_result* d_results, uint8_t* d_bits, void* cuda_stream);
MBE_B200_API int mbe_b200_process_indexed(mbe_b200_ctx* ctx, int codec, int input, const int32_t* slots, int n,
                                          int n_frames, const uint8_t* in, int16_t* pcm, float* pcmf,
                                          mbe_b200_result* results, uint8_t* bits);
MBE_B200_API int mbe_b200_submit_indexed(mbe_b200_ctx* ctx, int codec, int input, const int32_t* slots, int n, int n_frames,
                                         const uint8_t* in, int16_t* pcm, float* pcmf, mbe_b200_result* results,
                                         uint8_t* bits);
/* init_streams / export / import of the listed slots (host slot list; element i <-> slots[i] of the dense buffers) */
MBE_B200_API int mbe_b200_init_streams_indexed(mbe_b200_ctx* ctx, const int32_t* slots, int n, const uint32_t* seeds);
MBE_B200_API int mbe_b200_export_state_indexed(mbe_b200_ctx* ctx, const int32_t* slots, int n, void* parms_triplets);
MBE_B200_API int mbe_b200_import_state_indexed(mbe_b200_ctx* ctx, const int32_t* slots, int n, const void* parms_triplets);
MBE_B200_API int mbe_b200_export_rng_indexed(mbe_b200_ctx* ctx, const int32_t* slots, int n, uint32_t* rng_words4);
MBE_B200_API int mbe_b200_import_rng_indexed(mbe_b200_ctx* ctx, const int32_t* slots, int n, const uint32_t* rng_words4);

/* ---- stage-split entry points ----------------------------------------------------------------
 * decode_frames: batched mbe_decode<Codec>[Soft]Frame (mbelib.h:315,323,395,403,471,479,545,553):
 *   ECC + PN de-scrambling only; stateless; n = number of frames; bits [n][param_bits] one byte per bit.
 * process_data : batched mbe_process<Codec>Data / Dataf (mbelib.h:335-342, 415-419, 491-495): parameter
 *   bits -> PCM with the stream state; `results` is IN/OUT like the reference's result pointer (context
 *   flags C0_VALID/C4_VALID and counters in, status flags out); results==NULL means "no decode context"
 *   (the reference's result==NULL rules). IMBE 7100 uses the IMBE 4400 parameter layout (mbelib.h:545). */
MBE_B200_API int mbe_b200_decode_frames_dev(mbe_b200_ctx* ctx, int codec, int soft, int n, const uint8_t* d_frames,
                                            uint8_t* d_bits, mbe_b200_result* d_results, void* cuda_stream);
MBE_B200_API int mbe_b200_decode_frames(mbe_b200_ctx* ctx, int codec, int soft, int n, const uint8_t* frames,
                                        uint8_t* bits, mbe_b200_result* results);
/* ecc_blocks: batched mbe_golay2312 / mbe_golay2312Soft (code 0), mbe_hamming1511[Soft] (code 1) and
 *   mbe_7100x4400hamming1511[Soft] (code 2) (mbelib.h:238-274): n independent code words of 23 / 15 bits, one byte per
 *   bit with bit i of the word at index i (soft: mbe_soft_bit pairs); out = corrected word (Golay: corrected data bits,
 *   parity bits echoed from the input like the reference), status[i] = the reference's return value (changed data bits /
 *   corrected bits, or MBE_STATUS_INVALID_BITS with out[i] untouched). */
#define MBE_B200_ECC_GOLAY2312        0
#define MBE_B200_ECC_HAMMING1511      1
#define MBE_B200_ECC_HAMMING1511_7100 2
MBE_B200_API int mbe_b200_ecc_blocks_dev(mbe_b200_ctx* ctx, int code, int soft, int n, const uint8_t* d_in, uint8_t* d_out,
                                         int32_t* d_status, void* cuda_stream);
MBE_B200_API int mbe_b200_ecc_blocks(mbe_b200_ctx* ctx, int code, int soft, int n, const uint8_t* in, uint8_t* out,
                                     int32_t* status);
MBE_B200_API int mbe_b200_process_data_dev(mbe_b200_ctx* ctx, int codec, int first_stream, int n_streams, int n_frames,
                                           const uint8_t* d_bits, mbe_b200_result* d_results_inout, int16_t* d_pcm,
                                           float* d_pcmf, void* cuda_stream);
MBE_B200_API int mbe_b200_process_data(mbe_b200_ctx* ctx, int codec, int first_stream, int n_streams, int n_frames,
                                       const uint8_t* bits, mbe_b200_result* results_inout, int16_t* pcm, float* pcmf);
/* Indexed parameter-bit batches: process_data for any set of stream slots, the indexed calls above applied to
 * mbe_process<Codec>Data.  For a server whose frames arrive with the FEC already removed (P25 DFSI / ISSI carry IMBE as 88
 * information bits in 11 bytes), or that runs decode_frames itself before synthesis.
 *   - Element i is stream slot slots[i]: bits / results_inout / pcm / pcmf are laid out [i][frame][...] exactly like
 *     stream i of process_data, and every element consumes n_frames frames with the process_data rules above
 *     (results_inout IN/OUT, NULL = no decode context; IMBE 7100 takes the IMBE 4400 layout).
 *   - packed = 0: one byte per bit, as process_data; a byte other than 0 / 1 gives MBE_STATUS_INVALID_BITS (-2).
 *   - packed = 1: mbe_b200_packed_param_bytes(codec) = 11 / 11 / 7 / 7 bytes per frame, parameter bit k is bit
 *     7 - (k & 7) of byte k >> 3 (MSB first, as the packed channel frames); the pad bits of the last byte are ignored and
 *     MBE_STATUS_INVALID_BITS cannot occur.  A feed with another bit order is repacked by the caller.
 *   - Rejection: the rules of the indexed frame calls (out-of-range slot, or a repeat of a slot an earlier element names;
 *     the first occurrence wins; the whole list is checked, on the device for _dev).  A rejected element follows the rule
 *     of every negative status on this path, NOT the frame calls' zeroed result: each of its results is the caller's
 *     input element with only .status replaced by MBE_STATUS_INVALID_ARGUMENT (-1) (nothing is written when results_inout
 *     is NULL); its PCM and float PCM are zero and no stream state is touched.
 *   - n == 0 or n_frames == 0 returns 0 and launches nothing.  _dev / host / submit (completed by mbe_b200_wait) as for
 *     process_indexed[_dev] / submit_indexed: host calls refuse while a submission is pending, one submission may be
 *     pending per context, and concurrent calls whose slot sets overlap are the caller's error.
 * A contiguous caller that wants packed input passes the identity list first_stream .. first_stream + n - 1. */
MBE_B200_API int mbe_b200_packed_param_bytes(int codec);
MBE_B200_API int mbe_b200_process_data_indexed_dev(mbe_b200_ctx* ctx, int codec, int packed, const int32_t* d_slots, int n,
                                                   int n_frames, const uint8_t* d_bits, mbe_b200_result* d_results_inout,
                                                   int16_t* d_pcm, float* d_pcmf, void* cuda_stream);
MBE_B200_API int mbe_b200_process_data_indexed(mbe_b200_ctx* ctx, int codec, int packed, const int32_t* slots, int n,
                                               int n_frames, const uint8_t* bits, mbe_b200_result* results_inout,
                                               int16_t* pcm, float* pcmf);
MBE_B200_API int mbe_b200_submit_data_indexed(mbe_b200_ctx* ctx, int codec, int packed, const int32_t* slots, int n,
                                              int n_frames, const uint8_t* bits, mbe_b200_result* results_inout,
                                              int16_t* pcm, float* pcmf);

/* ---- single stages on caller-held parameter sets -------------------------------------------------------
 * Batched forms of the reference's per-stage helpers, one element = one call, host `mbe_parms` blobs updated in place:
 *   decode_parms         mbe_decodeImbe4400Parms / mbe_decodeAmbe2400Parms / mbe_decodeAmbe2450Parms (mbelib.h:301,385,461):
 *                        bits [n][88 or 49] -> cur[i] (w0, L, K, Vl, Ml, log2Ml, gamma) from prev[i]; prev[i] is updated
 *                        too (the decoders extend its magnitudes); status[i] = the reference's return value (0 voice,
 *                        codec-specific non-zero for invalid / erasure / tone frames, MBE_STATUS_INVALID_BITS).
 *   spectral_amp_enhance mbe_spectralAmpEnhance (mbelib.h:623); rm0 (optional) receives the pre-enhancement energy.
 *   adaptive_smoothing   mbe_applyAdaptiveSmoothing (mbelib.h:725).
 * They run the same device functions the frame kernels fuse and exist for stage-level consumers and stage-level parity. */
MBE_B200_API int mbe_b200_decode_parms(mbe_b200_ctx* ctx, int codec, int n, const uint8_t* bits, void* cur_parms,
                                       void* prev_parms, int32_t* status);
MBE_B200_API int mbe_b200_spectral_amp_enhance(mbe_b200_ctx* ctx, int n, void* cur_parms, float* rm0);
MBE_B200_API int mbe_b200_adaptive_smoothing(mbe_b200_ctx* ctx, int n, void* cur_parms, const void* prev_parms);
/*   synthesize_tone      mbe_synthesizeTonef (dstar_id == NULL: amplitude and tone index parsed from bits49) and
 *                        mbe_synthesizeTonefdstar (dstar_id[i] = ID1; bits49 may be NULL) (mbelib.h:630,638): 160 float
 *                        samples per element, cur[i]'s tone phases advanced; unknown tones and invalid bits give silence.
 *   comfort_noise        mbe_synthesizeComfortNoisef (mbelib.h:706) with the caller's RNG words (in/out, as export_rng).
 *   channel_step         the front-end one step at a time on caller-held frames, hard decision, one byte per bit:
 *                        step 0 mbe_ecc<Codec>C0 (frame in/out), 1 mbe_demodulate<Codec>Data (frame in/out),
 *                        2 mbe_ecc<Codec>Data (frame in, bits out), 3 mbe_convertImbe7100to7200 (bits in/out, codec 1 only);
 *                        status[i] = the reference's return value. */
MBE_B200_API int mbe_b200_synthesize_tone(mbe_b200_ctx* ctx, int n, const uint8_t* bits49, const int32_t* dstar_id,
                                          void* cur_parms, float* pcmf);
MBE_B200_API int mbe_b200_comfort_noise(mbe_b200_ctx* ctx, int n, uint32_t* rng_words4, float* pcmf);
MBE_B200_API int mbe_b200_channel_step(mbe_b200_ctx* ctx, int codec, int step, int n, uint8_t* frames, uint8_t* bits,
                                       int32_t* status);
/* ---- synthesis-only entry points --------------------------------------------------------------
 * synthesize_speech: batched mbe_synthesizeSpeechf / mbe_synthesizeSpeech (mbelib.h:652,662): element i
 *   synthesises one frame from host parameter sets cur[i], prev[i] (mbe_parms blobs, updated in place
 *   like the reference does) with RNG state as after mbe_setThreadRngSeed(seeds[i]) (seeds NULL: default).
 * floattoshort: batched mbe_floattoshort (mbelib.h:675), n_frames x 160 samples. */
MBE_B200_API int mbe_b200_synthesize_speech(mbe_b200_ctx* ctx, int n, void* cur_parms, void* prev_parms,
                                            const uint32_t* seeds, float* pcmf, int16_t* pcm);
/* the same with the RNG state carried by the caller: rng_words4 = [n][4] {comfort_seed48 lo, hi, unvoiced seed,
 * override flag} in and out, the words mbe_b200_export_rng moves (what the reference keeps in thread-local storage
 * between calls, src/core/mbe_adaptive.c:29-30, src/core/mbe_unvoiced_fft.c:29-30) */
MBE_B200_API int mbe_b200_synthesize_speech_rng(mbe_b200_ctx* ctx, int n, void* cur_parms, void* prev_parms,
                                                uint32_t* rng_words4, float* pcmf, int16_t* pcm);
MBE_B200_API int mbe_b200_floattoshort(mbe_b200_ctx* ctx, int n_frames, const float* in, int16_t* out);
MBE_B200_API int mbe_b200_floattoshort_dev(mbe_b200_ctx* ctx, int n_frames, const float* d_in, int16_t* d_out,
                                           void* cuda_stream);

/* ---- many GPUs from one process (SURVEY 8(e)) ------------------------------------------------------
 * A pool owns one context per device and shards the global stream range [0, max_streams) into contiguous blocks of
 * ceil(max_streams / n_devices) streams, block i on device_ordinals[i] (NULL: devices 0..n-1; n_devices == 0: every
 * visible device).  The same ordinal may be listed more than once (several contexts on one GPU).  A pool call runs the
 * corresponding per-context call on every shard that owns part of the stream range, concurrently from one host thread
 * per shard; all pointers are HOST pointers, laid out for the whole range exactly as in the per-context calls.  Nothing
 * is exchanged between GPUs (streams are independent): the host only scatters frame bits and gathers PCM.  End to end
 * the PCM gather is host-bandwidth bound on a many-GPU box (DESIGN.md section 6); keep PCM device-resident through
 * mbe_b200_pool_shard() + the _dev entry points when that matters. */
typedef struct mbe_b200_pool mbe_b200_pool;
MBE_B200_API int mbe_b200_pool_create(mbe_b200_pool** out, int n_devices, const int* device_ordinals, int max_streams);
MBE_B200_API void mbe_b200_pool_destroy(mbe_b200_pool* pool);
MBE_B200_API const char* mbe_b200_pool_last_error(const mbe_b200_pool* pool); /* pool may be NULL: last create() error */
MBE_B200_API int mbe_b200_pool_shards(const mbe_b200_pool* pool);
MBE_B200_API int mbe_b200_pool_shard(const mbe_b200_pool* pool, int shard, int* first_stream, int* n_streams,
                                     mbe_b200_ctx** ctx);
MBE_B200_API int mbe_b200_pool_init_streams(mbe_b200_pool* pool, int first_stream, int count, const uint32_t* seeds);
MBE_B200_API int mbe_b200_pool_export_state(mbe_b200_pool* pool, int first_stream, int count, void* parms_triplets);
MBE_B200_API int mbe_b200_pool_import_state(mbe_b200_pool* pool, int first_stream, int count, const void* parms_triplets);
MBE_B200_API int mbe_b200_pool_process_frames(mbe_b200_pool* pool, int codec, int soft, int first_stream, int n_streams,
                                              int n_frames, const uint8_t* frames, int16_t* pcm, float* pcmf,
                                              mbe_b200_result* results, uint8_t* bits);
/* Indexed pool calls: slots are global pool slots in [0, max_streams), laid out as in mbe_b200_process_indexed /
 * mbe_b200_init_streams_indexed.  Each shard gathers its elements (list order kept, so the first occurrence of a repeated
 * slot still wins), runs the context's indexed call on its local slots and scatters the outputs back; an out-of-range
 * element gets the rejected-element result of a context.  init_streams_indexed fails as a whole on a bad list. */
MBE_B200_API int mbe_b200_pool_process_indexed(mbe_b200_pool* pool, int codec, int input, const int32_t* slots, int n,
                                               int n_frames, const uint8_t* in, int16_t* pcm, float* pcmf,
                                               mbe_b200_result* results, uint8_t* bits);
/* mbe_b200_process_data_indexed over global pool slots, gathered and scattered the same way (the IN/OUT results travel
 * both ways); an out-of-range element gets the rejected-element result of the context call: the caller's result with
 * status -1, zero PCM. */
MBE_B200_API int mbe_b200_pool_process_data_indexed(mbe_b200_pool* pool, int codec, int packed, const int32_t* slots, int n,
                                                    int n_frames, const uint8_t* bits, mbe_b200_result* results_inout,
                                                    int16_t* pcm, float* pcmf);
MBE_B200_API int mbe_b200_pool_init_streams_indexed(mbe_b200_pool* pool, const int32_t* slots, int n, const uint32_t* seeds);
MBE_B200_API int mbe_b200_pool_set_channel_map(mbe_b200_pool* pool, int codec, const uint16_t* map, int n_bits);
MBE_B200_API int mbe_b200_pool_process_frames_packed(mbe_b200_pool* pool, int codec, int first_stream, int n_streams,
                                                     int n_frames, const uint8_t* packed, int16_t* pcm, float* pcmf,
                                                     mbe_b200_result* results, uint8_t* bits);
/* profiling aid: per-stage clock64() sums of the stream kernel; all zero unless the library was built with
 * -DMBE_STAGE_TIMING=1.  out16[0..7] = {frame barrier, front-end + decode, enhance + synthesis
 * setup, count barrier, voiced bank, unvoiced + hand-over, output stores, state store}, out16[8..13] = inside the bank
 * {oscillator setup, phase A, interpolation, wait A, phase B, wait B}; reset != 0 clears the counters. */
MBE_B200_API int mbe_b200_debug_stage_cycles(mbe_b200_ctx* ctx, unsigned long long* out16, int reset);

/* block until everything queued on the context's stream has finished */
MBE_B200_API int mbe_b200_synchronize(mbe_b200_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* MBE_B200_H */
