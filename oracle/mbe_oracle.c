/*
 * TEST INFRASTRUCTURE - CPU oracle (see mbe_oracle.h for scope and parity status: PINNED against
 * oracle/_ref/libmberef.so and the reference's golden vectors).
 *
 * Each section names the reference file:line whose behaviour it restates.  Floating-point
 * expressions keep the reference's evaluation order and float/double promotions; the file is built
 * with -ffp-contract=off (the reference's Release build targets SSE2, i.e. no FMA contraction).
 * libm calls go to the host glibc, as the reference's do.
 */
#define _GNU_SOURCE
#include "mbe_oracle.h"

#include <math.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#define MBE_TBL static const
#include "../mbelib-neo_b200/csrc/mbe_tables.inc"

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif
#ifndef M_SQRT2
#define M_SQRT2 1.41421356237309504880
#endif

#define NSAMP    160
#define FFTN     256
#define MAXBANDS 56

/* ============================================================================================
 * 0. small helpers
 * ========================================================================================== */

int
mbo_frame_bits(int codec) {
    return codec == MBO_IMBE7200 ? 184 : (codec == MBO_IMBE7100 ? 168 : 96);
}

int
mbo_param_bits(int codec) {
    return (codec == MBO_IMBE7200 || codec == MBO_IMBE7100) ? 88 : 49;
}

static int
bands_ok(int L) {
    return L >= 1 && L <= MAXBANDS;
}

static int
check_hard_bits(const char* b, size_t n) { /* src/internal/mbe_result.h:18-29 */
    if (!b) {
        return MBO_ERR_ARGUMENT;
    }
    for (size_t i = 0; i < n; ++i) {
        if (b[i] != 0 && b[i] != 1) {
            return MBO_ERR_BITS;
        }
    }
    return 0;
}

static int
check_soft_bits(const mbo_soft_bit* b, size_t n) { /* src/internal/mbe_result.h:31-42 */
    if (!b) {
        return MBO_ERR_ARGUMENT;
    }
    for (size_t i = 0; i < n; ++i) {
        if (b[i].bit > 1u) {
            return MBO_ERR_BITS;
        }
    }
    return 0;
}

/* ============================================================================================
 * 1. RNG state and parameter-state initialisation
 *    src/core/mbelib.c:173-181,367-410; src/core/mbe_adaptive.c:19-60; src/core/mbe_unvoiced_fft.c:295-302
 * ========================================================================================== */

#define LCG48_MUL  0x5DEECE66DULL
#define LCG48_ADD  0xBULL
#define LCG48_MASK ((1ULL << 48) - 1ULL)

void
mbo_rng_default(mbo_rng* rng) {
    rng->comfort_seed48 = (0x12345678ULL ^ LCG48_MUL) & LCG48_MASK;
    rng->uv_seed = 3147u;
    rng->uv_override = 0;
}

void
mbo_rng_seed(mbo_rng* rng, uint32_t seed) {
    if (seed == 0u) {
        seed = 0x6d25357bu;
    }
    rng->comfort_seed48 = (((uint64_t)seed) ^ LCG48_MUL) & LCG48_MASK;
    rng->uv_seed = seed % 53125u;
    rng->uv_override = 1;
}

static void
fill_default_model(mbo_parms* p, float w0, int L, int K, float mute_thr) {
    p->swn = 0;
    p->tonePhase = 0;
    p->w0 = w0;
    p->L = L;
    p->K = K;
    p->gamma = 0.0f;
    for (int l = 0; l <= 56; ++l) {
        p->Ml[l] = 1.0f;
        p->Vl[l] = 0;
        p->log2Ml[l] = 0.0f;
        p->PHIl[l] = 0.0f;
        p->PSIl[l] = 0.0f;
    }
    p->localEnergy = 75000.0f;
    p->amplitudeThreshold = 20480;
    p->errorRate = 0.0f;
    p->errorCountTotal = 0;
    p->errorCount4 = 0;
    p->repeatCount = 0;
    p->mutingThreshold = mute_thr;
    p->noiseSeed = -1.0f;
    memset(p->noiseOverlap, 0, sizeof(p->noiseOverlap));
    memset(p->previousUw, 0, sizeof(p->previousUw));
}

void
mbo_init_parms(mbo_parms* cur, mbo_parms* prev, mbo_parms* enh) { /* mbelib.c:367-410 */
    if (!cur || !prev || !enh) {
        return;
    }
    float w0 = (float)((4.0 * M_PI) / (134.0 + 39.5));
    int L = (int)(0.9254 * (int)((M_PI / w0) + 0.25));
    fill_default_model(prev, w0, L, 12, 0.0875f);
    *cur = *prev;
    *enh = *prev;
}

static void
init_ambe_parms(mbo_parms* cur, mbo_parms* prev, mbo_parms* enh) { /* ambe_common.c:191-229 */
    fill_default_model(prev, (float)((M_PI / 32.0) * (2.0 * M_PI)), 15, 0, 0.096f);
    *cur = *prev;
    *enh = *prev;
}

/* ============================================================================================
 * 2. ECC: Golay(23,12) and Hamming(15,11), hard and soft    (src/ecc/ecc.c)
 * ========================================================================================== */

static uint32_t
golay_parity_of_data(uint32_t data12) { /* XOR of generator rows of the set data bits, MSB first */
    uint32_t p = 0;
    for (int i = 0; i < 12; ++i) {
        if (data12 & (0x800u >> i)) {
            p ^= t_golay_gen[i];
        }
    }
    return p;
}

/* corrected 12 data bits of a received 23-bit word (ecc.c:221-251) */
static uint32_t
golay_correct_data(uint32_t w23) {
    uint32_t data = (w23 >> 11) & 0xfffu;
    uint32_t syn = golay_parity_of_data(data) ^ (w23 & 0x7ffu);
    return data ^ t_golay_fix[syn];
}

int
mbo_check_golay_block(long* block) {
    if (!block) {
        return MBO_ERR_ARGUMENT;
    }
    uint32_t b = (uint32_t)(*block);
    /* the reference does not mask the upper bits of `block >> 11` */
    uint32_t data = b >> 11;
    uint32_t syn = golay_parity_of_data((b >> 11) & 0xfffu) ^ (b & 0x7ffu);
    *block = (long)(int)(data ^ t_golay_fix[syn]);
    return 0;
}

static uint32_t
pack_bits_lsb0(const char* bits, int n) {
    uint32_t w = 0;
    for (int i = n - 1; i >= 0; --i) {
        w = (w << 1) | (uint32_t)(bits[i] & 1);
    }
    return w;
}

int
mbo_golay2312(const char* in, char* out) { /* ecc.c:259-301 */
    if (!out) {
        return MBO_ERR_ARGUMENT;
    }
    int rc = check_hard_bits(in, 23);
    if (rc < 0) {
        return rc;
    }
    uint32_t w = pack_bits_lsb0(in, 23);
    uint32_t fixed = golay_correct_data(w);
    for (int i = 0; i < 12; ++i) {
        out[11 + i] = (char)((fixed >> i) & 1u);
    }
    for (int i = 0; i < 11; ++i) {
        out[i] = in[i]; /* parity bits echo the input */
    }
    return __builtin_popcount(fixed ^ ((w >> 11) & 0xfffu));
}

/* lexicographic "candidate beats incumbent" rule of ecc.c:54-67 */
static int
soft_better(int have, int score, int best_score, int match, int best_match, int diffs, int best_diffs) {
    if (!have || score < best_score) {
        return 1;
    }
    if (score != best_score) {
        return 0;
    }
    if (match != best_match) {
        return match;
    }
    return diffs < best_diffs;
}

int
mbo_golay2312_soft(const mbo_soft_bit* in, char* out) { /* ecc.c:303-357 */
    if (!out) {
        return MBO_ERR_ARGUMENT;
    }
    int rc = check_soft_bits(in, 23);
    if (rc < 0) {
        return rc;
    }
    uint32_t hard = 0;
    for (int i = 22; i >= 0; --i) {
        hard = (hard << 1) | (uint32_t)(in[i].bit & 1u);
    }
    const uint32_t hard_fixed = golay_correct_data(hard);

    int have = 0, best_score = 0x3fffffff, best_diffs = 0x3fffffff, best_match = 0;
    uint32_t best_data = 0;
    for (uint32_t data = 0; data < 4096u; ++data) {
        uint32_t cw = (data << 11) | golay_parity_of_data(data);
        uint32_t diff = cw ^ hard;
        int score = 0;
        for (int i = 0; i < 23; ++i) {
            if ((diff >> i) & 1u) {
                score += (int)in[i].reliability;
            }
        }
        int diffs = __builtin_popcount(diff >> 11);
        int match = (data == hard_fixed);
        if (soft_better(have, score, best_score, match, have ? best_match : 0, diffs, best_diffs)) {
            best_data = data;
            best_score = score;
            best_diffs = diffs;
            best_match = match;
            have = 1;
        }
    }
    for (int i = 0; i < 12; ++i) {
        out[11 + i] = (char)((best_data >> i) & 1u);
    }
    for (int i = 0; i < 11; ++i) {
        out[i] = (char)(in[i].bit & 1u);
    }
    return best_diffs;
}

/* Hamming(15,11): two parity-check layouts (ecc_const.c:17-19). */
static const uint16_t ham_rows_std[4] = {0x7f08, 0x78e4, 0x66d2, 0x55b1};
static const uint16_t ham_rows_7100[4] = {0x7ac8, 0x3d64, 0x1eb2, 0x7591};
static const uint8_t ham_data_pos_std[11] = {2, 4, 5, 6, 8, 9, 10, 11, 12, 13, 14};
static const uint8_t ham_par_pos_std[4] = {0, 1, 3, 7};
static const uint8_t ham_data_pos_7100[11] = {4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14};
static const uint8_t ham_par_pos_7100[4] = {0, 1, 2, 3};

static int
ham_syndrome(uint32_t w15, const uint16_t rows[4]) {
    int s = 0;
    for (int i = 0; i < 4; ++i) {
        s |= (__builtin_popcount(w15 & rows[i]) & 1) << i;
    }
    return s;
}

/* syndrome -> single-bit flip mask: the bit whose parity-check column equals the syndrome.
 * Equals the reference's two 16-entry LUTs (ecc.c:28-36); syndromes with no matching column map to 0. */
static uint32_t
ham_flip_mask(int syn, const uint16_t rows[4]) {
    for (int b = 0; b < 15; ++b) {
        int col = 0;
        for (int i = 0; i < 4; ++i) {
            col |= ((rows[i] >> b) & 1) << i;
        }
        if (col == syn) {
            return 1u << b;
        }
    }
    return 0;
}

static uint32_t
ham_correct(uint32_t w15, const uint16_t rows[4], int* errs) {
    int syn = ham_syndrome(w15, rows);
    *errs = 0;
    if (syn > 0) {
        *errs = 1;
        w15 ^= ham_flip_mask(syn, rows);
    }
    return w15;
}

int
mbo_hamming1511(const char* in, char* out, int variant7100) { /* ecc.c:366-408,422-464 */
    if (!out) {
        return MBO_ERR_ARGUMENT;
    }
    int rc = check_hard_bits(in, 15);
    if (rc < 0) {
        return rc;
    }
    int errs;
    uint32_t w = ham_correct(pack_bits_lsb0(in, 15), variant7100 ? ham_rows_7100 : ham_rows_std, &errs);
    for (int i = 0; i < 15; ++i) {
        out[i] = (char)((w >> i) & 1u);
    }
    return errs;
}

int
mbo_hamming1511_soft(const mbo_soft_bit* in, char* out, int variant7100) { /* ecc.c:157-215 */
    if (!out) {
        return MBO_ERR_ARGUMENT;
    }
    int rc = check_soft_bits(in, 15);
    if (rc < 0) {
        return rc;
    }
    const uint16_t* rows = variant7100 ? ham_rows_7100 : ham_rows_std;
    const uint8_t* dpos = variant7100 ? ham_data_pos_7100 : ham_data_pos_std;
    const uint8_t* ppos = variant7100 ? ham_par_pos_7100 : ham_par_pos_std;

    uint32_t hard = 0;
    for (int i = 14; i >= 0; --i) {
        hard = (hard << 1) | (uint32_t)(in[i].bit & 1u);
    }
    int dummy;
    const uint32_t hard_fixed = ham_correct(hard, rows, &dummy);

    int have = 0, best_score = 0x3fffffff, best_diffs = 0x3fffffff;
    uint32_t best = 0;
    for (uint32_t data = 0; data < 2048u; ++data) {
        uint32_t cw = 0;
        for (int i = 0; i < 11; ++i) {
            cw |= ((data >> i) & 1u) << dpos[i];
        }
        int found = 0;
        for (int p = 0; p < 16 && !found; ++p) {
            uint32_t c = cw;
            for (int i = 0; i < 4; ++i) {
                c |= (uint32_t)((p >> i) & 1) << ppos[i];
            }
            if (ham_syndrome(c, rows) == 0) {
                cw = c;
                found = 1;
            }
        }
        if (!found) {
            continue;
        }
        uint32_t diff = cw ^ hard;
        int score = 0;
        for (int i = 0; i < 15; ++i) {
            if ((diff >> i) & 1u) {
                score += (int)in[i].reliability;
            }
        }
        int diffs = __builtin_popcount(diff);
        int match = (cw == hard_fixed);
        int best_match = have ? (best == hard_fixed) : 0;
        if (soft_better(have, score, best_score, match, best_match, diffs, best_diffs)) {
            best = cw;
            best_score = score;
            best_diffs = diffs;
            have = 1;
        }
    }
    if (!have) {
        best = hard_fixed;
        best_diffs = __builtin_popcount(best ^ hard);
    }
    for (int i = 0; i < 15; ++i) {
        out[i] = (char)((best >> i) & 1u);
    }
    return best_diffs;
}

/* ============================================================================================
 * 3. Codec front-ends: C0 ECC, PN de-scrambling, data ECC, parameter-bit packing
 *    src/imbe/imbe7200x4400.c:424-778, src/imbe/imbe7100x4400.c:99-516, src/ambe/ambe_common.c:22-189
 * ========================================================================================== */

typedef struct {
    uint8_t bit[8][24];
    uint8_t rel[8][24];
    int soft;
} frame_t;

/* one Golay row, hard or soft; `in`/`rel` length 23; writes the decoded bits back */
static int
golay_row(uint8_t* bits, const uint8_t* rel, int soft) {
    char out[23];
    int errs;
    if (soft) {
        mbo_soft_bit sb[23];
        for (int j = 0; j < 23; ++j) {
            sb[j].bit = bits[j];
            sb[j].reliability = rel[j];
        }
        errs = mbo_golay2312_soft(sb, out);
    } else {
        errs = mbo_golay2312((const char*)bits, out);
    }
    for (int j = 0; j < 23; ++j) {
        bits[j] = (uint8_t)(out[j] & 1);
    }
    return errs;
}

static int
hamming_row(uint8_t* bits, const uint8_t* rel, int soft, int v7100) {
    char out[15];
    int errs;
    if (soft) {
        mbo_soft_bit sb[15];
        for (int j = 0; j < 15; ++j) {
            sb[j].bit = bits[j];
            sb[j].reliability = rel[j];
        }
        errs = mbo_hamming1511_soft(sb, out, v7100);
    } else {
        errs = mbo_hamming1511((const char*)bits, out, v7100);
    }
    for (int j = 0; j < 15; ++j) {
        bits[j] = (uint8_t)(out[j] & 1);
    }
    return errs;
}

/* PN sequence: p0 = 16*seed, p(i) = (173 p(i-1) + 13849) mod 65536, output bit = p >> 15 */
static void
pn_bits(unsigned seed, int count, uint8_t* out /* out[1..count] */) {
    uint32_t p = (16u * seed) & 0xffffu;
    for (int i = 1; i <= count; ++i) {
        p = (173u * p + 13849u) & 0xffffu;
        out[i] = (uint8_t)(p >> 15);
    }
}

static int
decode_imbe7200(frame_t* f, char* d, mbo_result* r) {
    uint8_t pn[115];
    int c0 = golay_row(f->bit[0], f->rel[0], f->soft);

    unsigned seed = 0;
    for (int j = 22; j >= 11; --j) {
        seed = (seed << 1) | f->bit[0][j];
    }
    pn_bits(seed, 114, pn);
    int k = 1;
    for (int i = 1; i < 4; ++i) {
        for (int j = 22; j >= 0; --j) {
            f->bit[i][j] ^= pn[k++];
        }
    }
    for (int i = 4; i < 7; ++i) {
        for (int j = 14; j >= 0; --j) {
            f->bit[i][j] ^= pn[k++];
        }
    }

    int errs = 0, c4 = 0, o = 0;
    for (int j = 22; j > 10; --j) {
        d[o++] = (char)f->bit[0][j];
    }
    for (int i = 1; i < 4; ++i) {
        errs += golay_row(f->bit[i], f->rel[i], f->soft);
        for (int j = 22; j > 10; --j) {
            d[o++] = (char)f->bit[i][j];
        }
    }
    for (int i = 4; i < 7; ++i) {
        int e = hamming_row(f->bit[i], f->rel[i], f->soft, 0);
        errs += e;
        if (i == 4) {
            c4 = e;
        }
        for (int j = 14; j >= 4; --j) {
            d[o++] = (char)f->bit[i][j];
        }
    }
    for (int j = 6; j >= 0; --j) {
        d[o++] = (char)f->bit[7][j];
    }
    r->c0_errors = c0;
    r->protected_errors = errs;
    r->c4_errors = c4;
    r->total_errors = c0 + errs;
    r->flags = MBO_FLAG_C0_VALID | MBO_FLAG_C4_VALID | (f->soft ? MBO_FLAG_SOFT_INPUT : 0u);
    return c0 + errs;
}

/* 7100 -> 7200 parameter-bit permutation (imbe7100x4400.c:380-437) */
static void
imbe7100_to_7200(char* d) {
    static const uint8_t b0_idx[8] = {1, 2, 3, 4, 5, 6, 86, 87};
    int b0 = 0;
    for (int i = 0; i < 8; ++i) {
        b0 = (b0 << 1) | (d[b0_idx[i]] & 1);
    }
    float w0 = ((float)(4 * M_PI) / (float)((float)b0 + 39.5));
    int L = (int)(0.9254 * (int)((M_PI / w0) + 0.25));
    int K = (L < 37) ? (int)((float)(L + 2) / (float)3) : 12;

    char t[88];
    memset(t, 0, sizeof(t));
    t[87] = d[0];
    t[48 + K] = d[42];
    t[49 + K] = d[43];
    for (int i = 0; i < K; ++i) {
        t[48 + i] = d[44 + i];
    }
    int j = 0, k = 1;
    while (j < 87) {
        t[j] = d[k];
        if (++j == 48) {
            j += K + 2;
        }
        if (++k == 42) {
            k += K + 2;
        }
    }
    memcpy(d, t, 88);
}

static int
decode_imbe7100(frame_t* f, char* d, mbo_result* r) {
    uint8_t pn[115];
    uint8_t row[23], rel[23];
    /* C0: 18 received bits zero-extended to a 23-bit Golay word */
    for (int j = 0; j < 18; ++j) {
        row[j] = f->bit[0][j + 1];
        rel[j] = f->rel[0][j + 1];
    }
    for (int j = 18; j < 23; ++j) {
        row[j] = 0;
        rel[j] = 255;
    }
    int c0 = golay_row(row, rel, f->soft);
    for (int j = 0; j < 18; ++j) {
        f->bit[0][j + 1] = row[j];
    }

    unsigned seed = 0;
    for (int j = 18; j >= 12; --j) {
        seed = (seed << 1) | f->bit[0][j];
    }
    pn_bits(seed, 100, pn);
    int k = 1;
    for (int j = 23; j >= 0; --j) {
        f->bit[1][j] ^= pn[k++];
    }
    for (int i = 2; i < 4; ++i) {
        for (int j = 22; j >= 0; --j) {
            f->bit[i][j] ^= pn[k++];
        }
    }
    for (int i = 4; i < 6; ++i) {
        for (int j = 14; j >= 0; --j) {
            f->bit[i][j] ^= pn[k++];
        }
    }

    int errs = 0, c4 = 0, o = 0;
    for (int j = 18; j > 11; --j) {
        d[o++] = (char)f->bit[0][j];
    }
    errs = golay_row(&f->bit[1][1], &f->rel[1][1], f->soft); /* row 1 is offset by one column */
    for (int j = 22; j > 10; --j) {
        d[o++] = (char)f->bit[1][j + 1];
    }
    for (int i = 2; i < 4; ++i) {
        errs += golay_row(f->bit[i], f->rel[i], f->soft);
        for (int j = 22; j > 10; --j) {
            d[o++] = (char)f->bit[i][j];
        }
    }
    for (int i = 4; i < 6; ++i) {
        int e = hamming_row(f->bit[i], f->rel[i], f->soft, 1);
        errs += e;
        if (i == 4) {
            c4 = e;
        }
        for (int j = 14; j >= 4; --j) {
            d[o++] = (char)f->bit[i][j];
        }
    }
    for (int j = 22; j >= 0; --j) {
        d[o++] = (char)f->bit[6][j];
    }
    imbe7100_to_7200(d);
    r->c0_errors = c0;
    r->protected_errors = errs;
    r->c4_errors = c4;
    r->total_errors = c0 + errs;
    r->flags = MBO_FLAG_C0_VALID | MBO_FLAG_C4_VALID | (f->soft ? MBO_FLAG_SOFT_INPUT : 0u);
    return c0 + errs;
}

static int
decode_ambe3600(frame_t* f, char* d, mbo_result* r) {
    uint8_t pn[24];
    /* C0 = Golay(23,12) on columns 1..23 plus an overall parity bit in column 0 ("Golay24") */
    int c0 = golay_row(&f->bit[0][1], &f->rel[0][1], f->soft);
    if (c0 == 0) {
        int ones = 0;
        for (int j = 0; j < 24; ++j) {
            ones += f->bit[0][j];
        }
        if (ones & 1) {
            f->bit[0][0] ^= 1;
            c0 = 1;
        }
    }
    unsigned seed = 0;
    for (int j = 23; j >= 12; --j) {
        seed = (seed << 1) | f->bit[0][j];
    }
    pn_bits(seed, 23, pn);
    int k = 1;
    for (int j = 22; j >= 0; --j) {
        f->bit[1][j] ^= pn[k++];
    }
    int o = 0;
    for (int j = 23; j > 11; --j) {
        d[o++] = (char)f->bit[0][j];
    }
    int errs = golay_row(f->bit[1], f->rel[1], f->soft);
    for (int j = 22; j > 10; --j) {
        d[o++] = (char)f->bit[1][j];
    }
    for (int j = 10; j >= 0; --j) {
        d[o++] = (char)f->bit[2][j];
    }
    for (int j = 13; j >= 0; --j) {
        d[o++] = (char)f->bit[3][j];
    }
    r->c0_errors = c0;
    r->protected_errors = errs;
    r->c4_errors = 0;
    r->total_errors = c0 + errs;
    r->flags = MBO_FLAG_C0_VALID | (f->soft ? MBO_FLAG_SOFT_INPUT : 0u);
    return c0 + errs;
}

int
mbo_decode_frame(int codec, int soft, const void* frame, char* bits, mbo_result* result) {
    mbo_result local;
    if (result) {
        memset(result, 0, sizeof(*result));
    }
    if (!bits) {
        return MBO_ERR_ARGUMENT;
    }
    const int nbits = mbo_frame_bits(codec);
    const int cols = (codec == MBO_IMBE7200) ? 23 : 24;
    int rc = soft ? check_soft_bits((const mbo_soft_bit*)frame, (size_t)nbits)
                  : check_hard_bits((const char*)frame, (size_t)nbits);
    if (rc < 0) {
        return rc;
    }
    frame_t f;
    memset(&f, 0, sizeof(f));
    f.soft = soft;
    for (int i = 0; i < nbits; ++i) {
        if (soft) {
            f.bit[i / cols][i % cols] = ((const mbo_soft_bit*)frame)[i].bit & 1u;
            f.rel[i / cols][i % cols] = ((const mbo_soft_bit*)frame)[i].reliability;
        } else {
            f.bit[i / cols][i % cols] = (uint8_t)(((const char*)frame)[i] & 1);
        }
    }
    int ret;
    switch (codec) {
        case MBO_IMBE7200: ret = decode_imbe7200(&f, bits, &local); break;
        case MBO_IMBE7100: ret = decode_imbe7100(&f, bits, &local); break;
        default: ret = decode_ambe3600(&f, bits, &local); break;
    }
    if (result) {
        *result = local;
    }
    return ret;
}

/* ============================================================================================
 * 4. Parameter dequantisation
 * ========================================================================================== */

/* DCT cosine tables, built like the reference's lazily-filled caches: the argument is evaluated in
 * double and rounded to float on the cosf() call (imbe7200x4400.c:97-111, ambe3600x2450.c:60-74).
 *
 * One build-dependent detail of the parity target (the reference's default Release build, gcc -O3):
 * the compiler fully unrolls the 6x6 IMBE gain-DCT fill loop and folds its cosf() calls at compile
 * time, i.e. those 36 entries are CORRECTLY ROUNDED cosines, and two of them ([5][4], [5][6]) differ
 * by one ulp from what glibc's cosf() returns at run time.  (float)cos((double)x) reproduces the
 * folded values for all 36 arguments (checked against the compiled reference).  The 8x8 and the
 * per-block tables are filled at run time by glibc's cosf() in that build. */
typedef struct {
    int ready;
    float ri6[7][7];
    float ri8[9][9];
    float blk[18][18][18];
} dct_tables_t;

static dct_tables_t g_dct;
static pthread_once_t g_dct_once = PTHREAD_ONCE_INIT;

static void
dct_tables_fill(void) {
    for (int m = 1; m <= 6; ++m) {
        for (int i = 1; i <= 6; ++i) {
            float arg = (M_PI * (float)(m - 1) * ((float)i - 0.5f)) / 6.0f;
            g_dct.ri6[m][i] = (float)cos((double)arg);
        }
    }
    for (int m = 1; m <= 8; ++m) {
        for (int i = 1; i <= 8; ++i) {
            g_dct.ri8[m][i] = cosf((M_PI * (float)(m - 1) * ((float)i - 0.5f)) / 8.0f);
        }
    }
    for (int ji = 1; ji <= 17; ++ji) {
        for (int j = 1; j <= ji; ++j) {
            for (int k = 1; k <= ji; ++k) {
                g_dct.blk[ji][j][k] = cosf((M_PI * (float)(k - 1) * ((float)j - 0.5f)) / (float)ji);
            }
        }
    }
    g_dct.ready = 1;
}

static const dct_tables_t*
dct_tables(void) {
    pthread_once(&g_dct_once, dct_tables_fill);
    return &g_dct;
}

static int
bits_msb_first(const uint8_t* row, int hi) { /* value of row[hi..0], row[hi] most significant */
    int v = 0;
    for (int i = hi; i >= 0; --i) {
        v = (v << 1) | (row[i] & 1);
    }
    return v;
}

/* log-spectral-amplitude prediction shared by AMBE 2400/2450 (ambe3600x2450.c:389-459) */
static float
prev_log2(const mbo_parms* prev, int idx) {
    /* index 57 is one past log2Ml[]; in the reference's struct that address is PHIl[0] */
    return idx <= 56 ? prev->log2Ml[idx] : prev->PHIl[0];
}

/* ---- IMBE 4400 (imbe7200x4400.c:117-354,589-630) ---- */
int
mbo_decode_imbe4400_parms(const char* d, mbo_parms* cur, mbo_parms* prev) {
    if (!cur || !prev) {
        return MBO_ERR_ARGUMENT;
    }
    int rc = check_hard_bits(d, 88);
    if (rc < 0) {
        return rc;
    }
    static const uint8_t b0_idx[8] = {0, 1, 2, 3, 4, 5, 85, 86};
    int b0 = 0;
    for (int i = 0; i < 8; ++i) {
        b0 = (b0 << 1) | (d[b0_idx[i]] & 1);
    }
    if (b0 > 207) {
        return 1;
    }
    cur->w0 = ((float)(4 * M_PI) / (float)((float)b0 + 39.5));
    int L = (int)(0.9254 * (int)((M_PI / cur->w0) + 0.25));
    if (L > 56 || L < 9) {
        return 1;
    }
    cur->L = L;
    const int L9 = L - 9;
    cur->K = (L < 37) ? (int)((float)(L + 2) / (float)3) : 12;

    /* scatter bits 6..84 into per-parameter rows */
    uint8_t field[58][12];
    memset(field, 0, sizeof(field));
    const unsigned char* map = &t_imbe_bitmap[L9 * 79 * 2];
    for (int i = 6; i < 85; ++i) {
        field[map[0]][map[1]] = (uint8_t)d[i];
        map += 2;
    }

    /* V/UV: one decision per band of three harmonics, highest bit = lowest band */
    {
        int j = 1, k = cur->K - 1;
        for (int i = 1; i <= L; ++i) {
            cur->Vl[i] = (int)field[1][k];
            if (j == 3) {
                j = 1;
                if (k > 0) {
                    k--;
                }
            } else {
                j++;
            }
        }
    }

    /* gain vector */
    float Gm[7];
    Gm[1] = t_imbe_gain0[bits_msb_first(field[2], 5)];
    for (int i = 2; i < 7; ++i) {
        int nb = t_imbe_gain_bits[L9 * 5 + (i - 2)];
        float step = t_imbe_gain_step[L9 * 5 + (i - 2)];
        int bm = bits_msb_first(field[i + 1], nb - 1);
        Gm[i] = (step * ((float)bm - exp2f((float)nb - 1.0f) + 0.5f));
    }

    const dct_tables_t* T = dct_tables();
    float Ri[7];
    for (int i = 1; i <= 6; ++i) {
        float sum = 0;
        for (int m = 1; m <= 6; ++m) {
            int am = (m == 1) ? 1 : 2;
            sum = sum + ((float)am * Gm[m] * T->ri6[m][i]);
        }
        Ri[i] = sum;
    }

    /* higher-order DCT coefficients */
    float Cik[7][11];
    memset(Cik, 0, sizeof(Cik));
    {
        int m = 8;
        for (int i = 1; i <= 6; ++i) {
            Cik[i][1] = Ri[i];
            int ji = t_imbe_blocklen[L9 * 6 + (i - 1)];
            for (int k = 2; k <= ji; ++k) {
                int Bm = t_imbe_hoc_bits[L9 * 50 + (m - 8)];
                if (Bm <= 0) {
                    Cik[i][k] = 0;
                } else {
                    int bm = bits_msb_first(field[m], Bm - 1);
                    Cik[i][k] = ((t_imbe_hoc_step[Bm - 1] * t_imbe_hoc_sdev[k - 2])
                                 * (((float)bm - exp2f((float)Bm - 1.0f)) + 0.5f));
                }
                m++;
            }
        }
    }

    /* per-block inverse DCT */
    float Tl[57];
    memset(Tl, 0, sizeof(Tl));
    {
        int l = 1;
        for (int i = 1; i <= 6; ++i) {
            int ji = t_imbe_blocklen[L9 * 6 + (i - 1)];
            for (int j = 1; j <= ji; ++j) {
                float sum = 0;
                for (int k = 1; k <= ji; ++k) {
                    int ak = (k == 1) ? 1 : 2;
                    sum = sum + ((float)ak * Cik[i][k] * T->blk[ji][j][k]);
                }
                Tl[l++] = sum;
            }
        }
    }

    float rho;
    if (L <= 15) {
        rho = 0.4f;
    } else if (L <= 24) {
        rho = (0.03f * (float)L) - 0.05f;
    } else {
        rho = 0.7f;
    }

    /* prediction from the previous frame's log2 magnitudes */
    int cur_L = L;
    int prev_L = prev->L < 1 ? 1 : (prev->L > 56 ? 56 : prev->L);
    if (cur_L > prev_L) {
        for (int l = prev_L + 1; l <= cur_L; ++l) {
            prev->Ml[l] = prev->Ml[prev_L];
            prev->log2Ml[l] = prev->log2Ml[prev_L];
        }
    }
    prev->log2Ml[0] = prev->log2Ml[1];
    prev->Ml[0] = prev->Ml[1];

    int ik[57];
    float dl[57];
    float acc = 0;
    for (int l = 1; l <= cur_L; ++l) {
        float fk = ((float)prev_L / (float)cur_L) * (float)l;
        ik[l] = (int)fk;
        if (ik[l] < 0) {
            ik[l] = 0;
        } else if (ik[l] > 56) {
            ik[l] = 56;
        }
        dl[l] = fk - (float)ik[l];
        int up = ik[l] + 1 > 56 ? 56 : ik[l] + 1;
        acc = acc + ((((float)1 - dl[l]) * prev->log2Ml[ik[l]]) + (dl[l] * prev->log2Ml[up]));
    }
    acc = ((rho / (float)cur_L) * acc);
    for (int l = 1; l <= cur_L; ++l) {
        int up = ik[l] + 1 > 56 ? 56 : ik[l] + 1;
        float c1 = (rho * ((float)1 - dl[l]) * prev->log2Ml[ik[l]]);
        float c2 = (rho * dl[l] * prev->log2Ml[up]);
        cur->log2Ml[l] = Tl[l] + c1 + c2 - acc;
        cur->Ml[l] = exp2f(cur->log2Ml[l]);
    }
    return 0;
}

/* ---- shared AMBE tail: PRBA -> Ri -> Cik -> Tl -> magnitudes ---- */
typedef struct {
    const float* prba24; /* [512][3] */
    const float* prba58; /* [128][4] */
    const float* hoc[4]; /* [n][4]    */
    const unsigned char* blocklen; /* [57][4] */
} ambe_books_t;

static void
ambe_spectral_tail(mbo_parms* cur, mbo_parms* prev, const ambe_books_t* bk, int b3, int b4, const int hocidx[4],
                   float unvc) {
    const dct_tables_t* T = dct_tables();
    float Gm[9], Ri[9];
    Gm[1] = 0;
    Gm[2] = bk->prba24[b3 * 3 + 0];
    Gm[3] = bk->prba24[b3 * 3 + 1];
    Gm[4] = bk->prba24[b3 * 3 + 2];
    Gm[5] = bk->prba58[b4 * 4 + 0];
    Gm[6] = bk->prba58[b4 * 4 + 1];
    Gm[7] = bk->prba58[b4 * 4 + 2];
    Gm[8] = bk->prba58[b4 * 4 + 3];
    for (int i = 1; i <= 8; ++i) {
        float sum = 0;
        for (int m = 1; m <= 8; ++m) {
            int am = (m == 1) ? 1 : 2;
            sum = sum + ((float)am * Gm[m] * T->ri8[m][i]);
        }
        Ri[i] = sum;
    }

    const float rconst = ((float)1 / ((float)2 * M_SQRT2));
    float Cik[5][18];
    memset(Cik, 0, sizeof(Cik));
    int Ji[5];
    const int L = cur->L;
    for (int i = 1; i <= 4; ++i) {
        Cik[i][1] = (float)0.5 * (Ri[2 * i - 1] + Ri[2 * i]);
        Cik[i][2] = rconst * (Ri[2 * i - 1] - Ri[2 * i]);
        Ji[i] = bk->blocklen[L * 4 + (i - 1)];
        for (int k = 3; k <= Ji[i]; ++k) {
            Cik[i][k] = (k > 6) ? 0.0f : bk->hoc[i - 1][hocidx[i - 1] * 4 + (k - 3)];
        }
    }

    float Tl[57];
    memset(Tl, 0, sizeof(Tl));
    {
        int l = 1;
        for (int i = 1; i <= 4; ++i) {
            int ji = Ji[i];
            for (int j = 1; j <= ji; ++j) {
                float sum = 0;
                for (int k = 1; k <= ji; ++k) {
                    int ak = (k == 1) ? 1 : 2;
                    sum = sum + ((float)ak * Cik[i][k] * T->blk[ji][j][k]);
                }
                Tl[l++] = sum;
            }
        }
    }

    /* prediction (rho = 0.65) */
    int prev_L = prev->L;
    if (cur->L < 1) {
        cur->L = 1;
    } else if (cur->L > 56) {
        cur->L = 56;
    }
    if (prev_L < 1) {
        prev_L = 1;
    } else if (prev_L > 56) {
        prev_L = 56;
    }
    if (cur->L > prev_L) {
        for (int l = prev_L + 1; l <= cur->L; ++l) {
            prev->Ml[l] = prev->Ml[prev_L];
            prev->log2Ml[l] = prev->log2Ml[prev_L];
        }
    }
    prev->log2Ml[0] = prev->log2Ml[1];
    prev->Ml[0] = prev->Ml[1];

    int ik[57];
    float dl[57];
    float s43 = 0;
    for (int l = 1; l <= cur->L; ++l) {
        float fk = ((float)prev_L / (float)cur->L) * (float)l;
        ik[l] = (int)fk;
        dl[l] = fk - (float)ik[l];
        s43 = s43 + ((((float)1 - dl[l]) * prev_log2(prev, ik[l])) + (dl[l] * prev_log2(prev, ik[l] + 1)));
    }
    s43 = (((float)0.65 / (float)cur->L) * s43);

    float s42 = 0;
    for (int l = 1; l <= cur->L; ++l) {
        s42 += Tl[l];
    }
    s42 = s42 / (float)cur->L;
    float big_gamma = cur->gamma - (0.5f * log2f((float)cur->L)) - s42;

    for (int l = 1; l <= cur->L; ++l) {
        float c1 = ((float)0.65 * ((float)1 - dl[l]) * prev_log2(prev, ik[l]));
        float c2 = ((float)0.65 * dl[l] * prev_log2(prev, ik[l] + 1));
        cur->log2Ml[l] = Tl[l] + c1 + c2 - s43 + big_gamma;
        if (cur->Vl[l] == 1) {
            cur->Ml[l] = exp2f(cur->log2Ml[l]);
        } else {
            cur->Ml[l] = unvc * exp2f(cur->log2Ml[l]);
        }
    }
}

static int
pick_bits(const char* d, const uint8_t* idx, int n) {
    int v = 0;
    for (int i = 0; i < n; ++i) {
        v = (v << 1) | (d[idx[i]] & 1);
    }
    return v;
}

static int
tone_id_is_valid(int id) { /* src/internal/mbe_tone.h */
    return (id >= 5 && id <= 122) || (id >= 128 && id <= 163);
}

/* ---- AMBE+2 3600x2450 (ambe3600x2450.c:176-621) ---- */
int
mbo_decode_ambe2450_parms(const char* d, mbo_parms* cur, mbo_parms* prev, int total_errors) {
    if (!cur || !prev) {
        return MBO_ERR_ARGUMENT;
    }
    int rc = check_hard_bits(d, 49);
    if (rc < 0) {
        return rc;
    }
    static const uint8_t i_b0[7] = {0, 1, 2, 3, 37, 38, 39};
    static const uint8_t i_b1[5] = {4, 5, 6, 7, 35};
    static const uint8_t i_b2[5] = {8, 9, 10, 11, 36};
    static const uint8_t i_b3[9] = {12, 13, 14, 15, 16, 17, 18, 19, 40};
    static const uint8_t i_b4[7] = {20, 21, 22, 23, 41, 42, 43};
    static const uint8_t i_b5[5] = {24, 25, 26, 27, 44};
    static const uint8_t i_b6[4] = {28, 29, 30, 45};
    static const uint8_t i_b7[4] = {31, 32, 33, 46};
    static const uint8_t i_b8[3] = {34, 47, 48};

    /* tone classification on the four u-words */
    int u0 = 0, u1 = 0, u3 = 0;
    for (int i = 0; i < 12; ++i) {
        u0 = (u0 << 1) | d[i];
    }
    for (int i = 12; i < 24; ++i) {
        u1 = (u1 << 1) | d[i];
    }
    for (int i = 35; i < 49; ++i) {
        u3 = (u3 << 1) | d[i];
    }
    int tone_ok = (((u0 >> 6) & 0x3f) == 63) && (((u3 & 0xf) == 0) || (((u1 >> 8) & 0xf) == (u1 & 0xf)));
    if (tone_ok && total_errors < 6) {
        return 7;
    }

    int b0 = pick_bits(d, i_b0, 7);
    int silence = 0, L;
    float f0;
    if (b0 >= 120 && b0 <= 123) {
        return 2;
    }
    if (b0 == 124 || b0 == 125) {
        silence = 1;
        f0 = (float)M_PI / 32.0f;
        cur->w0 = f0 * (float)(2.0 * M_PI);
        L = (b0 == 124) ? 15 : 14;
        cur->L = L;
        for (int l = 1; l <= L; ++l) {
            cur->Vl[l] = 0;
        }
    } else if (b0 == 126 || b0 == 127) {
        return 2;
    } else {
        f0 = t_a2450_f0[b0];
        cur->w0 = f0 * (float)2 * M_PI;
        L = t_a2450_L[b0];
        cur->L = L;
    }

    float unvc = (float)0.2046 / sqrtf(cur->w0);

    int b1 = pick_bits(d, i_b1, 5);
    if (!silence) {
        for (int l = 1; l <= L; ++l) {
            int jl = (int)((float)l * (float)16.0 * f0);
            cur->Vl[l] = (t_a2450_vuv[b1] >> jl) & 1;
        }
    }
    int b2 = pick_bits(d, i_b2, 5);
    cur->gamma = t_a2450_dgain[b2] + ((float)0.5 * prev->gamma);

    ambe_books_t bk = {t_a2450_prba24, t_a2450_prba58, {t_a2450_hoc5, t_a2450_hoc6, t_a2450_hoc7, t_a2450_hoc8},
                       t_a2450_blocklen};
    int hocidx[4] = {pick_bits(d, i_b5, 5), pick_bits(d, i_b6, 4), pick_bits(d, i_b7, 4), pick_bits(d, i_b8, 3)};
    ambe_spectral_tail(cur, prev, &bk, pick_bits(d, i_b3, 9), pick_bits(d, i_b4, 7), hocidx, unvc);
    return 0;
}

/* ---- AMBE 3600x2400 (ambe3600x2400.c:164-546) ---- */
int
mbo_decode_ambe2400_parms(const char* d, mbo_parms* cur, mbo_parms* prev) {
    if (!cur || !prev) {
        return MBO_ERR_ARGUMENT;
    }
    int rc = check_hard_bits(d, 49);
    if (rc < 0) {
        return rc;
    }
    static const uint8_t i_b0[7] = {0, 1, 2, 3, 4, 5, 48};
    static const uint8_t i_b1[4] = {38, 39, 40, 41};
    static const uint8_t i_b2[6] = {6, 7, 8, 9, 42, 43};
    static const uint8_t i_b3[9] = {10, 11, 12, 13, 14, 15, 16, 44, 45};
    static const uint8_t i_b4[7] = {17, 18, 19, 20, 21, 46, 47};
    static const uint8_t i_b5[4] = {22, 23, 25, 26};
    static const uint8_t i_b6[4] = {27, 28, 29, 30};
    static const uint8_t i_b7[4] = {31, 32, 33, 34};
    static const uint8_t i_b8[3] = {35, 36, 37};

    int b0 = pick_bits(d, i_b0, 7);
    if ((b0 & 0x7E) == 0x7E) {
        /* tone index: three remapped high bits + five literal bits */
        static const uint8_t hi3[8] = {4, 0, 1, 2, 3, 7, 6, 5}; /* (t7<<2)|(t6<<1)|t5 per 3-bit selector */
        int sel = (d[6] << 2) | (d[7] << 1) | d[8];
        int tone = (hi3[sel] << 5) | (d[9] << 4) | (d[42] << 3) | (d[43] << 2) | (d[10] << 1) | d[11];
        if (tone >= 5 && tone <= 122) {
            return tone;
        }
        if (!(tone >= 128 && tone <= 163)) {
            cur->w0 = ((float)2 * M_PI) / (float)32;
            cur->L = 14;
            for (int l = 1; l <= 14; ++l) {
                cur->Vl[l] = 0;
            }
        }
        return 3;
    }

    float f0 = exp2f(-4.311767578125f - (2.1336e-2f * ((float)b0 + 0.5f)));
    cur->w0 = f0 * (float)2 * M_PI;
    int L = t_a2400_L[b0];
    cur->L = L;
    float unvc = (float)0.2046 / sqrtf(cur->w0);

    int b1 = pick_bits(d, i_b1, 4);
    for (int l = 1; l <= L; ++l) {
        int jl = (int)((float)l * (float)16.0 * f0);
        cur->Vl[l] = (t_a2400_vuv[b1] >> jl) & 1;
    }
    int b2 = pick_bits(d, i_b2, 6);
    cur->gamma = t_a2400_dgain[b2] + ((float)0.5 * prev->gamma);

    ambe_books_t bk = {t_a2400_prba24, t_a2400_prba58, {t_a2400_hoc5, t_a2400_hoc6, t_a2400_hoc7, t_a2400_hoc8},
                       t_a2400_blocklen};
    /* b8 is a 3-bit field stored in the upper bits of a 4-bit codebook index (LSB forced to 0) */
    int hocidx[4] = {pick_bits(d, i_b5, 4), pick_bits(d, i_b6, 4), pick_bits(d, i_b7, 4), pick_bits(d, i_b8, 3) << 1};
    ambe_spectral_tail(cur, prev, &bk, pick_bits(d, i_b3, 9), pick_bits(d, i_b4, 7), hocidx, unvc);
    return 0;
}

/* ============================================================================================
 * 5. Spectral amplitude enhancement and adaptive smoothing
 *    src/core/mbelib.c:412-661, src/core/mbe_adaptive.c:151-276
 * ========================================================================================== */

float
mbo_spectral_amp_enhance(mbo_parms* cur) {
    if (!cur || !bands_ok(cur->L)) {
        return 0.0f;
    }
    const int L = cur->L;
    float cosw[57];
    {
        float ss, cs;
        sincosf(cur->w0, &ss, &cs);
        float c = 1.0f, s = 0.0f;
        for (int l = 1; l <= L; ++l) {
            float cn = (c * cs) - (s * ss);
            float sn = (s * cs) + (c * ss);
            c = cn;
            s = sn;
            cosw[l] = c;
        }
    }
    float Rm0 = 0.0f, Rm1 = 0.0f;
    for (int l = 1; l <= L; ++l) {
        const float m2 = cur->Ml[l] * cur->Ml[l];
        Rm0 += m2;
        Rm1 += m2 * cosw[l];
    }
    const float R2m0 = Rm0 * Rm0;
    const float R2m1 = Rm1 * Rm1;
    for (int l = 1; l <= L; ++l) {
        if (cur->Ml[l] != 0.0f) {
            float W = sqrtf(cur->Ml[l])
                      * sqrtf(sqrtf(((float)0.96 * (float)M_PI * ((R2m0 + R2m1) - ((float)2 * Rm0 * Rm1 * cosw[l])))
                                    / (cur->w0 * Rm0 * (R2m0 - R2m1))));
            if ((8 * l) <= L) {
                /* low harmonics are left alone */
            } else if (W > 1.2f) {
                cur->Ml[l] = 1.2f * cur->Ml[l];
            } else if (W < 0.5f) {
                cur->Ml[l] = 0.5f * cur->Ml[l];
            } else {
                cur->Ml[l] = W * cur->Ml[l];
            }
        }
    }
    float sum = 0.0f;
    for (int l = 1; l <= L; ++l) {
        float M = cur->Ml[l];
        if (M < 0.0f) {
            M = -M;
        }
        sum += M * M;
    }
    float g = (sum == 0.0f) ? 1.0f : sqrtf(Rm0 / sum);
    for (int l = 1; l <= L; ++l) {
        cur->Ml[l] = g * cur->Ml[l];
    }
    return Rm0;
}

void
mbo_adaptive_smoothing(mbo_parms* cur, const mbo_parms* prev, int has_rm0, float rm0) {
    if (!cur || !prev || !bands_ok(cur->L) || !bands_ok(prev->L)) {
        return;
    }
    const int L = cur->L;
    if (!has_rm0) {
        rm0 = 0.0f;
        for (int l = 1; l <= L; ++l) {
            rm0 += cur->Ml[l] * cur->Ml[l];
        }
    }
    const float rate = cur->errorRate;
    const int etot = cur->errorCountTotal;
    const int e4 = cur->errorCount4;

    float pe = prev->localEnergy;
    if (pe < 10000.0f) {
        pe = 75000.0f;
    }
    float le = 0.95f * pe + 0.05f * rm0;
    if (le < 10000.0f) {
        le = 10000.0f;
    }
    cur->localEnergy = le;

    float VM;
    if (rate <= 0.005f && etot <= 4) {
        VM = __FLT_MAX__;
    } else {
        float x8 = sqrtf(sqrtf(sqrtf(le)));
        float en = x8 * x8 * x8;
        if (rate <= 0.0125f && e4 == 0) {
            VM = (45.255f * en) / expf(277.26f * rate);
        } else {
            VM = 1.414f * en;
        }
    }
    for (int l = 1; l <= L; ++l) {
        if (cur->Ml[l] > VM) {
            cur->Vl[l] = 1;
        }
    }
    float Am = 0.0f;
    for (int l = 1; l <= L; ++l) {
        Am += cur->Ml[l];
    }
    int pt = prev->amplitudeThreshold;
    if (pt <= 0) {
        pt = 20480;
    }
    int Tm;
    if (rate <= 0.005f && etot <= 6) {
        Tm = 20480;
    } else {
        Tm = 6000 - (300 * etot) + pt;
    }
    cur->amplitudeThreshold = Tm;
    if (Am > (float)Tm && Am > 0.0f) {
        float sc = (float)Tm / Am;
        for (int l = 1; l <= L; ++l) {
            cur->Ml[l] *= sc;
        }
    }
}

/* ============================================================================================
 * 6. Noise sources, 256-point real FFT, unvoiced synthesis
 *    src/core/mbe_unvoiced_fft.c, src/external/pffft/pffft.c (scalar N=256 path = FFTPACK radix-4)
 * ========================================================================================== */

void
mbo_comfort_noise(float* out, mbo_rng* rng) { /* mbe_adaptive.c:116-131 */
    const float gain = (0.003f * 32767.0f) / 7.0f;
    for (int i = 0; i < NSAMP; ++i) {
        rng->comfort_seed48 = (rng->comfort_seed48 * LCG48_MUL + LCG48_ADD) & LCG48_MASK;
        uint32_t r24 = (uint32_t)(rng->comfort_seed48 >> 24);
        float u = ((float)r24 / 16777216.0f) * 2.0f - 1.0f;
        out[i] = u * gain;
    }
}

void
mbo_noise_with_overlap(float* buf, float* seed, float* overlap, mbo_rng* rng) { /* mbe_unvoiced_fft.c:304-341 */
    if (*seed < 0.0f) {
        memset(buf, 0, FFTN * sizeof(float));
        memset(overlap, 0, 96 * sizeof(float));
        if (rng->uv_override) {
            *seed = (float)rng->uv_seed;
            rng->uv_override = 0;
        } else {
            *seed = 3147.0f;
        }
        return;
    }
    memcpy(buf, overlap, 96 * sizeof(float));
    unsigned st = ((unsigned)(*seed)) % 53125u;
    for (int i = 96; i < FFTN; ++i) {
        buf[i] = (float)st;
        st = (171u * st + 11213u) % 53125u;
    }
    *seed = (float)st;
    memcpy(overlap, buf + 160, 96 * sizeof(float));
}

/* twiddles exactly as FFTPACK's rffti1 computes them in the reference build: float angle, double
 * cos/sin, rounded to float (pffft.c:1231-1262) */
static float g_tw[FFTN];
static pthread_once_t g_tw_once = PTHREAD_ONCE_INIT;

static void
fft_twiddles_fill(void) {
    const int n = FFTN;
    float argh = (2 * M_PI) / n;
    int is = 0, l1 = 1;
    for (int pass = 1; pass <= 3; ++pass) { /* all four factors are 4; the last needs no twiddles */
        int l2 = l1 * 4;
        int ido = n / l2;
        int ld = 0;
        for (int j = 1; j <= 3; ++j) {
            int i = is, fi = 0;
            ld += l1;
            float argld = ld * argh;
            for (int ii = 3; ii <= ido; ii += 2) {
                i += 2;
                fi += 1;
                g_tw[i - 2] = cos(fi * argld);
                g_tw[i - 1] = sin(fi * argld);
            }
            is += ido;
        }
        l1 = l2;
    }
}

/* forward radix-4 butterfly stage: in is [4][l1][ido], out is [l1][4][ido] */
static void
rfft_fwd4(int ido, int l1, const float* in, float* out, const float* w1, const float* w2, const float* w3) {
#define IN(i, k, j)  in[(i) + ido * ((k) + l1 * (j))]
#define OUT(i, j, k) out[(i) + ido * ((j) + 4 * (k))]
    static const float nhs2 = (float)-0.7071067811865475;
    for (int k = 0; k < l1; ++k) {
        float a0 = IN(0, k, 0), a1 = IN(0, k, 1), a2 = IN(0, k, 2), a3 = IN(0, k, 3);
        float tr1 = a1 + a3;
        float tr2 = a0 + a2;
        OUT(ido - 1, 1, k) = a0 - a2;
        OUT(0, 2, k) = a3 - a1;
        OUT(0, 0, k) = tr1 + tr2;
        OUT(ido - 1, 3, k) = tr2 - tr1;
    }
    if (ido < 2) {
        return;
    }
    if (ido != 2) {
        for (int k = 0; k < l1; ++k) {
            for (int i = 2; i < ido; i += 2) {
                int ic = ido - i;
                float cr2 = IN(i - 1, k, 1), ci2 = IN(i, k, 1);
                float cr3 = IN(i - 1, k, 2), ci3 = IN(i, k, 2);
                float cr4 = IN(i - 1, k, 3), ci4 = IN(i, k, 3);
                float t;
                /* multiply by conj(w) */
                t = cr2 * w1[i - 1];
                cr2 = (cr2 * w1[i - 2]) + (ci2 * w1[i - 1]);
                ci2 = (ci2 * w1[i - 2]) - t;
                t = cr3 * w2[i - 1];
                cr3 = (cr3 * w2[i - 2]) + (ci3 * w2[i - 1]);
                ci3 = (ci3 * w2[i - 2]) - t;
                t = cr4 * w3[i - 1];
                cr4 = (cr4 * w3[i - 2]) + (ci4 * w3[i - 1]);
                ci4 = (ci4 * w3[i - 2]) - t;

                float x0r = IN(i - 1, k, 0), x0i = IN(i, k, 0);
                float tr1 = cr2 + cr4, tr4 = cr4 - cr2;
                float tr2 = x0r + cr3, tr3 = x0r - cr3;
                OUT(i - 1, 0, k) = tr1 + tr2;
                OUT(ic - 1, 3, k) = tr2 - tr1;
                float ti1 = ci2 + ci4, ti4 = ci2 - ci4;
                OUT(i - 1, 2, k) = ti4 + tr3;
                OUT(ic - 1, 1, k) = tr3 - ti4;
                float ti2 = x0i + ci3, ti3 = x0i - ci3;
                OUT(i, 0, k) = ti1 + ti2;
                OUT(ic, 3, k) = ti1 - ti2;
                OUT(i, 2, k) = tr4 + ti3;
                OUT(ic, 1, k) = tr4 - ti3;
            }
        }
        if (ido % 2 == 1) {
            return;
        }
    }
    for (int k = 0; k < l1; ++k) {
        float a = IN(ido - 1, k, 1), b = IN(ido - 1, k, 3);
        float c = IN(ido - 1, k, 0), d = IN(ido - 1, k, 2);
        float ti1 = nhs2 * (a + b);
        float tr1 = nhs2 * (b - a);
        OUT(ido - 1, 0, k) = tr1 + c;
        OUT(ido - 1, 2, k) = c - tr1;
        OUT(0, 1, k) = ti1 - d;
        OUT(0, 3, k) = ti1 + d;
    }
#undef IN
#undef OUT
}

/* backward radix-4 stage: in is [l1][4][ido], out is [4][l1][ido] */
static void
rfft_bwd4(int ido, int l1, const float* in, float* out, const float* w1, const float* w2, const float* w3) {
#define IN(i, j, k)  in[(i) + ido * ((j) + 4 * (k))]
#define OUT(i, k, j) out[(i) + ido * ((k) + l1 * (j))]
    static const float nsq2 = (float)-1.414213562373095;
    for (int k = 0; k < l1; ++k) {
        float a = IN(0, 0, k), b = IN(ido - 1, 3, k), c = IN(0, 2, k), d = IN(ido - 1, 1, k);
        float tr3 = 2.f * d;
        float tr2 = a + b;
        float tr1 = a - b;
        float tr4 = 2.f * c;
        OUT(0, k, 0) = tr2 + tr3;
        OUT(0, k, 2) = tr2 - tr3;
        OUT(0, k, 1) = tr1 - tr4;
        OUT(0, k, 3) = tr1 + tr4;
    }
    if (ido < 2) {
        return;
    }
    if (ido != 2) {
        for (int k = 0; k < l1; ++k) {
            for (int i = 2; i < ido; i += 2) {
                int ic = ido - i;
                float tr1 = IN(i - 1, 0, k) - IN(ic - 1, 3, k);
                float tr2 = IN(i - 1, 0, k) + IN(ic - 1, 3, k);
                float ti4 = IN(i - 1, 2, k) - IN(ic - 1, 1, k);
                float tr3 = IN(i - 1, 2, k) + IN(ic - 1, 1, k);
                OUT(i - 1, k, 0) = tr2 + tr3;
                float cr3 = tr2 - tr3;
                float ti3 = IN(i, 2, k) - IN(ic, 1, k);
                float tr4 = IN(i, 2, k) + IN(ic, 1, k);
                float cr2 = tr1 - tr4;
                float cr4 = tr1 + tr4;
                float ti1 = IN(i, 0, k) + IN(ic, 3, k);
                float ti2 = IN(i, 0, k) - IN(ic, 3, k);
                OUT(i, k, 0) = ti2 + ti3;
                float ci3 = ti2 - ti3;
                float ci2 = ti1 + ti4;
                float ci4 = ti1 - ti4;
                float t;
                t = cr2 * w1[i - 1];
                cr2 = (cr2 * w1[i - 2]) - (ci2 * w1[i - 1]);
                ci2 = (ci2 * w1[i - 2]) + t;
                OUT(i - 1, k, 1) = cr2;
                OUT(i, k, 1) = ci2;
                t = cr3 * w2[i - 1];
                cr3 = (cr3 * w2[i - 2]) - (ci3 * w2[i - 1]);
                ci3 = (ci3 * w2[i - 2]) + t;
                OUT(i - 1, k, 2) = cr3;
                OUT(i, k, 2) = ci3;
                t = cr4 * w3[i - 1];
                cr4 = (cr4 * w3[i - 2]) - (ci4 * w3[i - 1]);
                ci4 = (ci4 * w3[i - 2]) + t;
                OUT(i - 1, k, 3) = cr4;
                OUT(i, k, 3) = ci4;
            }
        }
        if (ido % 2 == 1) {
            return;
        }
    }
    for (int k = 0; k < l1; ++k) {
        float c = IN(ido - 1, 0, k), d = IN(ido - 1, 2, k);
        float a = IN(0, 1, k), b = IN(0, 3, k);
        float tr1 = c - d;
        float tr2 = c + d;
        float ti1 = b + a;
        float ti2 = b - a;
        OUT(ido - 1, k, 0) = tr2 + tr2;
        OUT(ido - 1, k, 1) = nsq2 * (ti1 - tr1);
        OUT(ido - 1, k, 2) = ti2 + ti2;
        OUT(ido - 1, k, 3) = nsq2 * (ti1 + tr1);
    }
#undef IN
#undef OUT
}

/* forward transform; output in "ordered" layout [DC, Nyquist, re1, im1, ...] (pffft.c:2019-2043) */
void
mbo_fft256_forward_ordered(const float* in, float* out) {
    pthread_once(&g_tw_once, fft_twiddles_fill);
    float a[FFTN], b[FFTN];
    rfft_fwd4(1, 64, in, a, g_tw + 252, g_tw + 253, g_tw + 254);
    rfft_fwd4(4, 16, a, b, g_tw + 240, g_tw + 244, g_tw + 248);
    rfft_fwd4(16, 4, b, a, g_tw + 192, g_tw + 208, g_tw + 224);
    rfft_fwd4(64, 1, a, b, g_tw + 0, g_tw + 64, g_tw + 128);
    out[0] = b[0];
    out[1] = b[FFTN - 1];
    for (int k = 2; k < FFTN; ++k) {
        out[k] = b[k - 1];
    }
}

void
mbo_fft256_backward_ordered(const float* in, float* out) {
    pthread_once(&g_tw_once, fft_twiddles_fill);
    float a[FFTN], b[FFTN];
    a[0] = in[0];
    a[FFTN - 1] = in[1];
    for (int k = 1; k < FFTN - 1; ++k) {
        a[k] = in[k + 1];
    }
    rfft_bwd4(64, 1, a, b, g_tw + 0, g_tw + 64, g_tw + 128);
    rfft_bwd4(16, 4, b, a, g_tw + 192, g_tw + 208, g_tw + 224);
    rfft_bwd4(4, 16, a, b, g_tw + 240, g_tw + 244, g_tw + 248);
    rfft_bwd4(1, 64, b, out, g_tw + 252, g_tw + 253, g_tw + 254);
}

static float
uv_window(int n) { /* n in [-105,105], else 0 */
    return (n < -105 || n > 105) ? 0.0f : t_win_unvoiced[n + 105];
}

static void
unvoiced_synthesis(float* out, mbo_parms* cur, const mbo_parms* prev, const float* noise) {
    /* mbe_unvoiced_fft.c:714-761 */
    if (!bands_ok(cur->L) || !bands_ok(prev->L)) {
        return;
    }
    float Uw[FFTN], F[FFTN], Uo[FFTN], scale[FFTN / 2 + 1];
    memset(scale, 0, sizeof(scale));
    for (int i = 0; i < FFTN; ++i) {
        Uw[i] = noise[i] * uv_window(i - 128);
    }
    mbo_fft256_forward_ordered(Uw, F);

    const float mult = (256.0f / (2.0f * 3.14159265358979323846f)) * cur->w0;
    for (int l = 1; l <= cur->L; ++l) {
        int a = (int)ceilf((l - 0.5f) * mult);
        int b = (int)ceilf((l + 0.5f) * mult);
        if (a < 0) {
            a = 0;
        }
        if (b > FFTN / 2) {
            b = FFTN / 2;
        }
        if (cur->Vl[l] != 0) {
            continue;
        }
        /* band energy over bins [a,b) in bin order; bin 0 has no imaginary part */
        float num = 0.0f;
        if (b > a) {
            int s = a;
            if (s == 0) {
                num += F[0] * F[0];
                s = 1;
            }
            for (int bin = s; bin < b; ++bin) {
                float re = F[2 * bin], im = F[2 * bin + 1];
                num += (re * re) + (im * im);
            }
        }
        int cnt = b - a;
        if (cnt > 0 && num > 1e-10f) {
            float sc = 146.17696f * cur->Ml[l] / sqrtf(num / (float)cnt);
            for (int bin = a; bin < b; ++bin) {
                scale[bin] = sc;
            }
        }
    }
    F[0] *= scale[0];
    for (int bin = 1; bin < FFTN / 2; ++bin) {
        F[2 * bin] *= scale[bin];
        F[2 * bin + 1] *= scale[bin];
    }
    F[1] *= scale[FFTN / 2];

    mbo_fft256_backward_ordered(F, Uo);
    const float inv = 1.0f / (float)FFTN;
    for (int i = 0; i < FFTN; ++i) {
        Uo[i] *= inv;
    }

    /* weighted overlap-add with the previous frame's inverse transform */
    for (int n = 0; n < NSAMP; ++n) {
        float wp = uv_window(n), wc = uv_window(n - NSAMP);
        float den = (wp * wp) + (wc * wc);
        float ps = (n + 128 < FFTN) ? prev->previousUw[n + 128] : 0.0f;
        float cs = (n - 32 >= 0 && n - 32 < FFTN) ? Uo[n - 32] : 0.0f;
        if (den > 1e-10f) {
            out[n] += ((wp * ps) + (wc * cs)) / den;
        }
    }
    memcpy(cur->previousUw, Uo, sizeof(Uo));
}

/* ============================================================================================
 * 7. Voiced synthesis and the per-frame synthesis orchestrator   (src/core/mbelib.c:895-1105)
 * ========================================================================================== */

#define TWO_PI_F (2.0f * (float)M_PI)
#define CLIP_F   ((32767.0f * 0.95f) / 7.0f)

/* mbo_run_work: where the frame being decoded by this thread reports its oscillator-bank work (null: nowhere) */
static __thread int32_t* g_work;

static void
voiced_windowed(float* out, const float* W, float gain, float phase0, float step) {
    float sd, cd, s, c;
    sincosf(step, &sd, &cd);
    sincosf(phase0, &s, &c);
    for (int n = 0; n < NSAMP; ++n) {
        out[n] += gain * W[n] * c;
        float cn = (c * cd) - (s * sd);
        float sn = (s * cd) + (c * sd);
        c = cn;
        s = sn;
    }
}

void
mbo_synthesize_speech(float* out, mbo_parms* cur, mbo_parms* prev, int has_rm0, float rm0, mbo_rng* rng) {
    const int N = NSAMP;
    if (!out) {
        return;
    }
    if (!cur || !prev || !bands_ok(cur->L) || !bands_ok(prev->L)) {
        memset(out, 0, N * sizeof(float));
        return;
    }
    mbo_adaptive_smoothing(cur, prev, has_rm0, rm0);

    int mute_on_rate = (fabsf(cur->mutingThreshold - 0.096f) > 1e-6f);
    if (cur->repeatCount >= 4 || (mute_on_rate && cur->errorRate > cur->mutingThreshold)) {
        mbo_comfort_noise(out, rng);
        return;
    }

    float noise[FFTN];
    mbo_noise_with_overlap(noise, &cur->noiseSeed, cur->noiseOverlap, rng);
    memset(out, 0, N * sizeof(float));

    /* bands present in only one of the two frames fade in/out as zero-amplitude voiced bands */
    int maxl;
    if (cur->L > prev->L) {
        maxl = cur->L;
        for (int l = prev->L + 1; l <= maxl; ++l) {
            prev->Ml[l] = 0.0f;
            prev->Vl[l] = 1;
        }
    } else {
        maxl = prev->L;
        for (int l = cur->L + 1; l <= maxl; ++l) {
            cur->Ml[l] = 0.0f;
            cur->Vl[l] = 1;
        }
    }

    int numUv = 0;
    for (int l = 0; l <= cur->L; ++l) {
        if (cur->Vl[l] == 0) {
            numUv++;
        }
    }

    int n_slots = 0, n_interp = 0;   /* the frame's work on the device's oscillator bank (mbo_run_work) */
    const float cw0 = cur->w0, pw0 = prev->w0;
    for (int l = 1; l <= 56; ++l) {
        float wrapped = fmodf(prev->PSIl[l], TWO_PI_F);
        if (wrapped < 0.0f) {
            wrapped += TWO_PI_F;
        }
        prev->PSIl[l] = wrapped;
        cur->PSIl[l] = wrapped + ((pw0 + cw0) * ((float)(l * N) / 2.0f));
        if (l <= (cur->L / 4)) {
            cur->PHIl[l] = cur->PSIl[l];
        } else {
            float pl = ((2.0f * (float)M_PI / 53125.0f) * noise[l]) - (float)M_PI;
            cur->PHIl[l] = cur->PSIl[l] + (((float)numUv * pl) / (float)cur->L);
        }
    }

    for (int l = 1; l <= maxl; ++l) {
        float cw0l = cw0 * (float)l;
        float pw0l = pw0 * (float)l;
        int cv = (cur->Vl[l] == 1), pv = (prev->Vl[l] == 1);
        if (!cv && !pv) {
            continue;
        }
        if ((l < 8) && cv && pv && (fabsf(cw0 - pw0) < (0.1f * cw0))) {
            n_slots++;
            n_interp++;
            /* phase/amplitude interpolation for stable low harmonics */
            float dphi = cur->PHIl[l] - prev->PHIl[l] - (((pw0 + cw0) * (float)(l * N)) / 2.0f);
            float dw = (1.0f / (float)N)
                       * (dphi - (2.0f * (float)M_PI * floorf((dphi + (float)M_PI) / (2.0f * (float)M_PI))));
            for (int n = 0; n < N; ++n) {
                float th = prev->PHIl[l] + ((pw0l + dw) * (float)n)
                           + (((cw0 - pw0) * (float)(l * n * n)) / (float)(2 * N));
                float a = prev->Ml[l] + (((float)n / (float)N) * (cur->Ml[l] - prev->Ml[l]));
                out[n] += 2.0f * a * cosf(th);
            }
        } else {
            /* a windowed component of gain exactly 0 adds +-0 and gets no slot, unless its phase is not finite (its
             * product is NaN then) */
            n_slots += (pv && ((2.0f * prev->Ml[l]) != 0.0f || !isfinite(prev->PHIl[l])))
                       + (cv && ((2.0f * cur->Ml[l]) != 0.0f || !isfinite(cur->PHIl[l])));
            /* the reference adds prev then cur per sample; the two contributions go to the same
             * accumulator in that order, which is what two sequential passes would NOT give when
             * both are present - so interleave them explicitly */
            if (pv && cv) {
                float sdp, cdp, sp, cp, sdc, cdc, sc, cc;
                const float gp = 2.0f * prev->Ml[l], gc = 2.0f * cur->Ml[l];
                sincosf(pw0l, &sdp, &cdp);
                sincosf(prev->PHIl[l], &sp, &cp);
                sincosf(cw0l, &sdc, &cdc);
                sincosf(cur->PHIl[l] - (cw0l * (float)N), &sc, &cc);
                for (int n = 0; n < N; ++n) {
                    out[n] += gp * t_win_voiced[n + N] * cp;
                    out[n] += gc * t_win_voiced[n] * cc;
                    float t1 = (cp * cdp) - (sp * sdp);
                    float t2 = (sp * cdp) + (cp * sdp);
                    cp = t1;
                    sp = t2;
                    t1 = (cc * cdc) - (sc * sdc);
                    t2 = (sc * cdc) + (cc * sdc);
                    cc = t1;
                    sc = t2;
                }
            } else if (pv) {
                voiced_windowed(out, t_win_voiced + N, 2.0f * prev->Ml[l], prev->PHIl[l], pw0l);
            } else {
                voiced_windowed(out, t_win_voiced, 2.0f * cur->Ml[l], cur->PHIl[l] - (cw0l * (float)N), cw0l);
            }
        }
    }
    if (g_work) {
        g_work[0] = n_slots;
        g_work[1] = n_interp;
        g_work[2] = 1;
    }

    unvoiced_synthesis(out, cur, prev, noise);

    for (int n = 0; n < N; ++n) {
        if (out[n] > CLIP_F) {
            out[n] = CLIP_F;
        } else if (out[n] < -CLIP_F) {
            out[n] = -CLIP_F;
        }
    }
}

/* ============================================================================================
 * 8. Tone synthesis, float -> int16                     (src/core/mbelib.c:692-856,1148-1177)
 * ========================================================================================== */

static int
tone_freqs(int id, float* f1, float* f2) { /* src/internal/mbe_tone.h:15-59 */
    static const float dual[36][2] = {
        {1336, 941}, {1209, 697}, {1336, 697}, {1477, 697}, {1209, 770}, {1336, 770}, {1477, 770}, {1209, 852},
        {1336, 852}, {1477, 852}, {1633, 697}, {1633, 770}, {1633, 852}, {1633, 941}, {1209, 941}, {1477, 941},
        {1162, 820}, {1052, 606}, {1162, 606}, {1279, 606}, {1052, 672}, {1162, 672}, {1279, 672}, {1052, 743},
        {1162, 743}, {1279, 743}, {1430, 606}, {1430, 672}, {1430, 743}, {1430, 820}, {1052, 820}, {1279, 820},
        {440, 350},  {480, 440},  {620, 480},  {490, 350}};
    *f1 = *f2 = 0.0f;
    if (id == 5) {
        *f1 = *f2 = 156.25f;
        return 1;
    }
    if (id == 6) {
        *f1 = *f2 = 187.5f;
        return 1;
    }
    if (id >= 7 && id <= 122) {
        *f1 = *f2 = 31.25f * (float)id;
        return 1;
    }
    if (id >= 128 && id <= 163) {
        *f1 = dual[id - 128][0];
        *f2 = dual[id - 128][1];
        return 1;
    }
    return 0;
}

static uint32_t
tone_step(double hz) {
    double st = (hz / 8000.0) * 4294967296.0;
    return st <= 0.0 ? 0u : (uint32_t)(st + 0.5);
}

static float
tone_sample(uint32_t phase) {
    float ang = (float)(((double)phase * ((2.0 * M_PI) / 4294967296.0)) - (M_PI / 2.0));
    return sinf(ang);
}

static void
render_tone(float* out, mbo_parms* cur, float f1, float f2, int amp) {
    if (!out) {
        return;
    }
    if (!cur || f1 <= 0.0f) {
        memset(out, 0, NSAMP * sizeof(float));
        return;
    }
    const int dual = (f2 > 0.0f) && (fabsf(f2 - f1) > 1e-6f);
    const float gain = (((amp < 0) ? 0.0f : (float)amp) / 127.0f) * CLIP_F;
    const uint32_t s1 = tone_step((double)f1);
    const uint32_t s2 = dual ? tone_step((double)f2) : 0u;
    uint32_t p1 = (uint32_t)cur->swn, p2 = cur->tonePhase;
    for (int n = 0; n < NSAMP; ++n) {
        p1 += s1;
        float a = tone_sample(p1);
        if (dual) {
            p2 += s2;
            float b = tone_sample(p2);
            out[n] = (0.5f * gain * a) + (0.5f * gain * b);
        } else {
            out[n] = gain * a;
        }
    }
    cur->swn = (int)p1;
    cur->tonePhase = p2;
}

void
mbo_synthesize_tone(float* out, const char* d, mbo_parms* cur) { /* mbelib.c:745-804 */
    if (!out) {
        return;
    }
    if (!cur || check_hard_bits(d, 49) < 0) {
        memset(out, 0, NSAMP * sizeof(float));
        return;
    }
    int u0 = 0, u1 = 0, u3 = 0;
    for (int i = 0; i < 12; ++i) {
        u0 = (u0 << 1) | d[i];
    }
    for (int i = 12; i < 24; ++i) {
        u1 = (u1 << 1) | d[i];
    }
    for (int i = 35; i < 49; ++i) {
        u3 = (u3 << 1) | d[i];
    }
    int AD = ((u0 & 0x3f) << 1) + ((u3 >> 4) & 0x1);
    int ID1 = ((u1 & 0xfff) >> 4);
    float f1, f2;
    if (!tone_freqs(ID1, &f1, &f2)) {
        memset(out, 0, NSAMP * sizeof(float));
        return;
    }
    render_tone(out, cur, f1, f2, AD);
}

void
mbo_synthesize_tone_dstar(float* out, mbo_parms* cur, int id1) { /* mbelib.c:813-856 */
    float f1 = 0;
    if (!out) {
        return;
    }
    if (!cur) {
        memset(out, 0, NSAMP * sizeof(float));
        return;
    }
    if (id1 == 5) {
        f1 = 156.25f;
    } else if (id1 == 6) {
        f1 = 187.5f;
    } else if (id1 >= 7 && id1 <= 122) {
        f1 = 31.25f * (float)id1;
    }
    if (f1 <= 0.0f) {
        memset(out, 0, NSAMP * sizeof(float));
        return;
    }
    render_tone(out, cur, f1, f1, 103);
}

void
mbo_float_to_short(const float* in, short* out) { /* mbelib.c:1148-1177,1312-1320 */
    const float maxa = 32767.0f * 0.95f;
    for (int i = 0; i < NSAMP; ++i) {
        uint32_t u;
        memcpy(&u, &in[i], 4);
        uint32_t a = u & 0x7fffffffu;
        float v;
        if (a > 0x7f800000u) {
            v = 0.0f;
        } else if (a == 0x7f800000u) {
            v = (u >> 31) ? -maxa : maxa;
        } else {
            v = 7.0f * in[i];
            if (v > maxa) {
                v = maxa;
            } else if (v < -maxa) {
                v = -maxa;
            }
        }
        out[i] = (short)v;
    }
}

/* ============================================================================================
 * 9. Per-frame state machines: parameter bits -> PCM
 *    imbe7200x4400.c:780-909, ambe3600x2450.c:716-898, ambe3600x2400.c:629-762, ambe_common.c:231-271
 * ========================================================================================== */

#define CONTEXT_FLAGS (MBO_FLAG_SOFT_INPUT | MBO_FLAG_C0_VALID | MBO_FLAG_C4_VALID)
#define STATUS_FLAGS  (MBO_FLAG_TONE | MBO_FLAG_ERASURE | MBO_FLAG_REPEAT | MBO_FLAG_MUTE)

static int
count_ok(int c) {
    return c >= 0 && c <= 184;
}

/* src/internal/mbe_result.h:44-97 */
static int
resolve_total_errors(const mbo_result* r, int* total) {
    *total = 0;
    if (!r) {
        return 0;
    }
    if ((r->flags & ~(CONTEXT_FLAGS | STATUS_FLAGS)) != 0u) {
        return MBO_ERR_ARGUMENT;
    }
    if (!count_ok(r->c0_errors) || !count_ok(r->protected_errors) || !count_ok(r->c4_errors)
        || !count_ok(r->total_errors)) {
        return MBO_ERR_ARGUMENT;
    }
    if (r->c0_errors > 184 - r->protected_errors) {
        return MBO_ERR_ARGUMENT;
    }
    int comp = r->c0_errors + r->protected_errors;
    if (!count_ok(comp)) {
        return MBO_ERR_ARGUMENT;
    }
    int t = (r->total_errors == 0 && comp != 0) ? comp : r->total_errors;
    int c0v = (r->flags & MBO_FLAG_C0_VALID) != 0u, c4v = (r->flags & MBO_FLAG_C4_VALID) != 0u;
    if (!((comp == 0 || t == comp) && (!c0v || t >= r->c0_errors) && (!c4v || t >= r->c4_errors))) {
        return MBO_ERR_ARGUMENT;
    }
    *total = t;
    return 0;
}

static void
prepare_result(mbo_result* r, int total) { /* mbe_result.h:99-114 */
    if (!r) {
        return;
    }
    unsigned ctx = r->flags & CONTEXT_FLAGS;
    int c0 = (ctx & MBO_FLAG_C0_VALID) ? r->c0_errors : 0;
    int c4 = (ctx & MBO_FLAG_C4_VALID) ? r->c4_errors : 0;
    r->flags = ctx;
    r->c0_errors = c0;
    r->c4_errors = c4;
    r->total_errors = total;
    r->protected_errors = total - c0;
}

static void
voice_frame(float* out, mbo_parms* cur, mbo_parms* prev, mbo_parms* enh, mbo_rng* rng) {
    *prev = *cur;
    float rm0 = mbo_spectral_amp_enhance(cur);
    mbo_synthesize_speech(out, cur, enh, 1, rm0, rng);
    *enh = *cur;
}

static int
process_imbe(float* out, mbo_result* r, const char* d, mbo_parms* cur, mbo_parms* prev, mbo_parms* enh,
             mbo_rng* rng) {
    int total;
    int rc = resolve_total_errors(r, &total);
    if (rc < 0) {
        return rc;
    }
    rc = check_hard_bits(d, 88);
    if (rc < 0) {
        return rc;
    }
    int c0v = (r->flags & MBO_FLAG_C0_VALID) != 0u, c4v = (r->flags & MBO_FLAG_C4_VALID) != 0u;
    int c0 = c0v ? r->c0_errors : 0;
    cur->errorCount4 = c4v ? r->c4_errors : 0;
    prepare_result(r, total);
    cur->mutingThreshold = 0.0875f;
    cur->errorCountTotal = total;
    cur->errorRate = (0.95f * prev->errorRate) + (0.000365f * (float)total);

    int bad = mbo_decode_imbe4400_parms(d, cur, prev);
    if (bad < 0) {
        return bad;
    }
    float thr = 10.0f + (40.0f * cur->errorRate);
    int repeat;
    if (bad == 1) {
        repeat = 1;
    } else if (c0v) {
        repeat = (c0 >= 2) && ((float)total >= thr);
    } else {
        repeat = total > 5;
    }
    if (!repeat) {
        cur->repeatCount = 0;
    } else {
        if (prev->repeatCount > 3) {
            /* headroom exhausted: fall back to the default voice model, keep continuity state */
            cur->swn = 0;
            cur->tonePhase = 0;
            cur->w0 = (float)((4.0 * M_PI) / (134.0 + 39.5));
            cur->L = (int)(0.9254 * (int)((M_PI / cur->w0) + 0.25));
            cur->K = 12;
            cur->gamma = 0.0f;
            for (int l = 0; l <= 56; ++l) {
                cur->Vl[l] = 0;
                cur->Ml[l] = 1.0f;
                cur->log2Ml[l] = 0.0f;
            }
            cur->repeatCount = 0;
            cur->localEnergy = 75000.0f;
            cur->amplitudeThreshold = 20480;
            cur->mutingThreshold = 0.0875f;
        } else {
            *cur = *prev;
            cur->repeatCount++;
        }
        r->flags |= MBO_FLAG_REPEAT;
    }
    int muted = (cur->repeatCount >= 4) || (cur->errorRate > cur->mutingThreshold);
    voice_frame(out, cur, prev, enh, rng);
    if (muted) {
        r->flags |= MBO_FLAG_MUTE;
    }
    return r->total_errors;
}

static void
set_erasure_model(mbo_parms* mp, const mbo_parms* src) { /* ambe_common.c:231-260 */
    mp->swn = 0;
    mp->tonePhase = 0;
    mp->w0 = 0.0f;
    mp->L = 9;
    mp->K = 0;
    mp->gamma = 0.0f;
    for (int l = 0; l <= 56; ++l) {
        mp->Ml[l] = 1.0f;
        mp->Vl[l] = 0;
        mp->log2Ml[l] = 0.0f;
        mp->PHIl[l] = src->PHIl[l];
        mp->PSIl[l] = src->PSIl[l];
    }
    mp->localEnergy = 75000.0f;
    mp->amplitudeThreshold = 20480;
    mp->noiseSeed = src->noiseSeed;
    memcpy(mp->noiseOverlap, src->noiseOverlap, sizeof(mp->noiseOverlap));
    memcpy(mp->previousUw, src->previousUw, sizeof(mp->previousUw));
}

static int
prepare_ambe(mbo_result* r, const char* d, mbo_parms* cur, mbo_parms* prev, mbo_parms* enh, int* total, int* c0,
             int* c0v) {
    int rc = resolve_total_errors(r, total);
    if (rc < 0) {
        return rc;
    }
    rc = check_hard_bits(d, 49);
    if (rc < 0) {
        return rc;
    }
    *c0v = (r->flags & MBO_FLAG_C0_VALID) != 0u;
    *c0 = *c0v ? r->c0_errors : 0;
    prepare_result(r, *total);
    if (fabsf(prev->mutingThreshold - 0.096f) > 1e-6f) {
        init_ambe_parms(cur, prev, enh); /* first AMBE frame after a generic init */
    }
    cur->mutingThreshold = 0.096f;
    cur->errorCountTotal = *total;
    cur->errorCount4 = 0;
    cur->errorRate = (0.95f * prev->errorRate) + (0.001064f * (float)cur->errorCountTotal);
    return 0;
}

static void
ambe_voice_or_mute(float* out, mbo_result* r, mbo_parms* cur, mbo_parms* prev, mbo_parms* enh, mbo_rng* rng) {
    if (cur->repeatCount < 4) {
        voice_frame(out, cur, prev, enh, rng);
        return;
    }
    r->flags |= MBO_FLAG_MUTE;
    mbo_comfort_noise(out, rng);
    init_ambe_parms(cur, prev, enh);
}

static int
process_ambe2450(float* out, mbo_result* r, const char* d, mbo_parms* cur, mbo_parms* prev, mbo_parms* enh,
                 mbo_rng* rng) {
    int total, c0, c0v;
    int rc = prepare_ambe(r, d, cur, prev, enh, &total, &c0, &c0v);
    if (rc < 0) {
        return rc;
    }
    int bad = mbo_decode_ambe2450_parms(d, cur, prev, total);
    if (bad < 0) {
        return bad;
    }
    /* decode-state update */
    if (bad == 2) {
        r->flags |= MBO_FLAG_ERASURE;
        cur->repeatCount = 0;
        set_erasure_model(cur, prev);
    } else if (bad == 3 || bad == 7) {
        r->flags |= MBO_FLAG_TONE;
        cur->repeatCount = 0;
    } else {
        int repeat = c0v ? ((c0 >= 4) || ((c0 >= 2) && (total >= 6))) : (total > 3);
        if (repeat) {
            *cur = *prev;
            cur->repeatCount++;
            r->flags |= MBO_FLAG_REPEAT;
        } else {
            cur->repeatCount = 0;
        }
    }
    /* synthesis */
    if (bad == 0) {
        ambe_voice_or_mute(out, r, cur, prev, enh, rng);
    } else if (bad == 7) {
        int id1 = 0;
        for (int i = 12; i < 20; ++i) {
            id1 = (id1 << 1) | (int)d[i];
        }
        if (tone_id_is_valid(id1)) {
            mbo_synthesize_tone(out, d, cur);
        } else if (!(prev->repeatCount >= 4)) {
            /* invalid tone id: replay the last voice model while advancing synthesis state */
            mbo_parms tmp = *enh;
            mbo_synthesize_speech(out, &tmp, enh, 0, 0.0f, rng);
            *enh = tmp;
        } else {
            mbo_comfort_noise(out, rng);
            init_ambe_parms(cur, prev, enh);
        }
    } else if (bad == 2) {
        mbo_comfort_noise(out, rng);
        *prev = *cur;
        *enh = *cur;
    } else {
        mbo_comfort_noise(out, rng);
        init_ambe_parms(cur, prev, enh);
    }
    return r->total_errors;
}

static int
process_ambe2400(float* out, mbo_result* r, const char* d, mbo_parms* cur, mbo_parms* prev, mbo_parms* enh,
                 mbo_rng* rng) {
    int total, c0, c0v;
    int rc = prepare_ambe(r, d, cur, prev, enh, &total, &c0, &c0v);
    if (rc < 0) {
        return rc;
    }
    int bad = mbo_decode_ambe2400_parms(d, cur, prev);
    if (bad < 0) {
        return bad;
    }
    const int clean_tone = (bad >= 7) && (bad <= 122) && (c0 < 2) && (total < 3);
    if (bad == 2) {
        r->flags |= MBO_FLAG_ERASURE;
        cur->repeatCount = 0;
        set_erasure_model(cur, prev);
    } else if (bad == 3) {
        r->flags |= MBO_FLAG_TONE;
        cur->repeatCount = 0;
    } else if (clean_tone) {
        /* state untouched */
    } else if (total > 3) {
        *cur = *prev;
        cur->repeatCount++;
        r->flags |= MBO_FLAG_REPEAT;
    } else {
        cur->repeatCount = 0;
    }

    if (clean_tone) {
        mbo_synthesize_tone_dstar(out, cur, bad);
        *prev = *cur;
    } else if (bad == 0) {
        ambe_voice_or_mute(out, r, cur, prev, enh, rng);
    } else if (bad == 2) {
        mbo_comfort_noise(out, rng);
        *prev = *cur;
        *enh = *cur;
    } else {
        mbo_comfort_noise(out, rng);
        init_ambe_parms(cur, prev, enh);
    }
    return r->total_errors;
}

int
mbo_process_data(int codec, float* out, mbo_result* result, const char* bits, mbo_parms* cur, mbo_parms* prev,
                 mbo_parms* enh, mbo_rng* rng) {
    mbo_result local;
    if (!result) {
        memset(&local, 0, sizeof(local));
        result = &local;
    }
    if (!out || !cur || !prev || !enh || !rng) {
        return MBO_ERR_ARGUMENT;
    }
    switch (codec) {
        case MBO_IMBE7200:
        case MBO_IMBE7100: return process_imbe(out, result, bits, cur, prev, enh, rng);
        case MBO_AMBE2400: return process_ambe2400(out, result, bits, cur, prev, enh, rng);
        case MBO_AMBE2450: return process_ambe2450(out, result, bits, cur, prev, enh, rng);
        default: return MBO_ERR_ARGUMENT;
    }
}

int
mbo_process_frame(int codec, int soft, float* out, mbo_result* result, const void* frame, char* bits, mbo_parms* cur,
                  mbo_parms* prev, mbo_parms* enh, mbo_rng* rng) {
    mbo_result local;
    if (!result) {
        result = &local;
    }
    int ret = mbo_decode_frame(codec, soft, frame, bits, result);
    if (ret < 0) {
        return ret;
    }
    return mbo_process_data(codec, out, result, bits, cur, prev, enh, rng);
}

/* ============================================================================================
 * 10. Batch driver (same contract as oracle/ref_bench.c)
 * ========================================================================================== */

typedef struct {
    int codec, soft, n_streams, n_frames, stride, nthreads, tid;
    const uint8_t* frames;
    const uint32_t* seeds;
    int16_t* pcm;
    float* pcmf;
    int32_t* results;
    uint8_t* bits;
    mbo_parms* state;
    int32_t* work;
} run_t;

static void*
run_worker(void* arg) {
    run_t* j = (run_t*)arg;
    const int fb = mbo_frame_bits(j->codec);
    const int pb = mbo_param_bits(j->codec);
    const size_t fstride = (size_t)fb * (j->soft ? 2u : 1u);
    for (int s = j->tid; s < j->n_streams; s += j->nthreads) {
        mbo_parms cur, prev, enh;
        mbo_rng rng;
        mbo_rng_default(&rng);
        mbo_rng_seed(&rng, j->seeds ? j->seeds[s] : 0u);
        mbo_init_parms(&cur, &prev, &enh);
        for (int f = 0; f < j->n_frames; ++f) {
            const size_t idx = (size_t)s * j->n_frames + f;
            const uint8_t* fr = j->frames + idx * fstride;
            char d[88];
            float pf[NSAMP];
            short ps[NSAMP];
            mbo_result res;
            memset(d, 0, sizeof(d));
            memset(&res, 0, sizeof(res));
            if (j->work) {
                g_work = j->work + idx * 3;
                memset(g_work, 0, 3 * sizeof(int32_t));
            }
            int ret = mbo_process_frame(j->codec, j->soft, pf, &res, fr, d, &cur, &prev, &enh, &rng);
            g_work = NULL;
            if (ret < 0) {
                memset(pf, 0, sizeof(pf));
                memset(ps, 0, sizeof(ps));
            } else {
                mbo_float_to_short(pf, ps);
            }
            if (j->pcm) {
                memcpy(j->pcm + idx * NSAMP, ps, sizeof(ps));
            }
            if (j->pcmf) {
                memcpy(j->pcmf + idx * NSAMP, pf, sizeof(pf));
            }
            if (j->results) {
                int32_t* r = j->results + idx * 6;
                r[0] = ret;
                r[1] = res.c0_errors;
                r[2] = res.protected_errors;
                r[3] = res.c4_errors;
                r[4] = res.total_errors;
                r[5] = (int32_t)res.flags;
            }
            if (j->bits) {
                memcpy(j->bits + idx * pb, d, (size_t)pb);
            }
        }
        if (j->state) {
            j->state[(size_t)s * 3 + 0] = cur;
            j->state[(size_t)s * 3 + 1] = prev;
            j->state[(size_t)s * 3 + 2] = enh;
        }
    }
    return NULL;
}

double
mbo_run(int codec, int soft, int n_streams, int n_frames, const uint8_t* frames, const uint32_t* seeds, int16_t* pcm,
        float* pcmf, int32_t* results, uint8_t* bits, void* state, int n_threads) {
    return mbo_run_work(codec, soft, n_streams, n_frames, frames, seeds, pcm, pcmf, results, bits, state, NULL, n_threads);
}

double
mbo_run_work(int codec, int soft, int n_streams, int n_frames, const uint8_t* frames, const uint32_t* seeds, int16_t* pcm,
             float* pcmf, int32_t* results, uint8_t* bits, void* state, int32_t* work, int n_threads) {
    if (n_threads < 1) {
        n_threads = 1;
    }
    if (n_threads > 256) {
        n_threads = 256;
    }
    (void)dct_tables();
    pthread_once(&g_tw_once, fft_twiddles_fill);
    run_t jobs[256];
    pthread_t th[256];
    struct timespec t0, t1;
    clock_gettime(CLOCK_MONOTONIC, &t0);
    for (int t = 0; t < n_threads; ++t) {
        run_t j = {codec, soft, n_streams, n_frames, 0, n_threads, t, frames, seeds, pcm, pcmf, results, bits,
                   (mbo_parms*)state, work};
        jobs[t] = j;
        if (n_threads > 1) {
            pthread_create(&th[t], NULL, run_worker, &jobs[t]);
        }
    }
    if (n_threads == 1) {
        run_worker(&jobs[0]);
    } else {
        for (int t = 0; t < n_threads; ++t) {
            pthread_join(th[t], NULL);
        }
    }
    clock_gettime(CLOCK_MONOTONIC, &t1);
    return (double)(t1.tv_sec - t0.tv_sec) + 1e-9 * (double)(t1.tv_nsec - t0.tv_nsec);
}

/* ---- batched block decoders (threaded): what tests/test_gpu_ecc_blocks.py compares mbe_b200_ecc_blocks with ---------- */
/* code: 0 Golay(23,12), 1 Hamming(15,11), 2 Hamming(15,11) in the IMBE 7100 layout; in: [n][len] bits or [n][len] soft-bit
 * pairs; out: [n][len]; status[i] = the decoder's return value.
 * fast != 0 (soft only): the same exhaustive search - every data word in ascending order, the same (score, equals the hard
 * decode, differing bits) triple, the same soft_better() rule - with the code words from a table built once and the score
 * from three per-word byte tables instead of a 23-step loop (~40x faster, so a million words per code finish in seconds).
 * tests/test_oracle_kat.py checks it word for word against mbo_golay2312_soft / mbo_hamming1511_soft. */
static uint32_t g_golay_cw[4096];
static uint16_t g_ham_cw[2][2048];
static pthread_once_t g_cw_once = PTHREAD_ONCE_INIT;

static void
cw_tables_fill(void) {
    for (uint32_t d = 0; d < 4096u; ++d) {
        g_golay_cw[d] = (d << 11) | golay_parity_of_data(d);
    }
    for (int v = 0; v < 2; ++v) {
        const uint16_t* rows = v ? ham_rows_7100 : ham_rows_std;
        const uint8_t* dpos = v ? ham_data_pos_7100 : ham_data_pos_std;
        const uint8_t* ppos = v ? ham_par_pos_7100 : ham_par_pos_std;
        for (uint32_t data = 0; data < 2048u; ++data) {
            uint32_t cw = 0;
            for (int i = 0; i < 11; ++i) {
                cw |= ((data >> i) & 1u) << dpos[i];
            }
            for (int p = 0; p < 16; ++p) {
                uint32_t c = cw;
                for (int i = 0; i < 4; ++i) {
                    c |= (uint32_t)((p >> i) & 1) << ppos[i];
                }
                if (ham_syndrome(c, rows) == 0) {
                    cw = c;
                    break;
                }
            }
            g_ham_cw[v][data] = (uint16_t)cw; /* (every data word has a parity completion) */
        }
    }
}

static void
score_tables(const mbo_soft_bit* in, int len, int tab[3][256]) {
    for (int g = 0; g < 3; ++g) {
        for (int x = 0; x < 256; ++x) {
            int sc = 0;
            for (int b = 0; b < 8; ++b) {
                const int i = 8 * g + b;
                if (i < len && ((x >> b) & 1)) {
                    sc += (int)in[i].reliability;
                }
            }
            tab[g][x] = sc;
        }
    }
}

static int
golay_soft_fast(const mbo_soft_bit* in, char* out) {
    int rc = check_soft_bits(in, 23);
    if (rc < 0) {
        return rc;
    }
    uint32_t hard = 0;
    for (int i = 22; i >= 0; --i) {
        hard = (hard << 1) | (uint32_t)(in[i].bit & 1u);
    }
    const uint32_t hard_fixed = golay_correct_data(hard);
    int tab[3][256];
    score_tables(in, 23, tab);
    int have = 0, best_score = 0x3fffffff, best_diffs = 0x3fffffff, best_match = 0;
    uint32_t best_data = 0;
    for (uint32_t data = 0; data < 4096u; ++data) {
        const uint32_t diff = g_golay_cw[data] ^ hard;
        const int score = tab[0][diff & 255u] + tab[1][(diff >> 8) & 255u] + tab[2][diff >> 16];
        const int diffs = __builtin_popcount(diff >> 11);
        const int match = (data == hard_fixed);
        if (soft_better(have, score, best_score, match, have ? best_match : 0, diffs, best_diffs)) {
            best_data = data;
            best_score = score;
            best_diffs = diffs;
            best_match = match;
            have = 1;
        }
    }
    for (int i = 0; i < 12; ++i) {
        out[11 + i] = (char)((best_data >> i) & 1u);
    }
    for (int i = 0; i < 11; ++i) {
        out[i] = (char)(in[i].bit & 1u);
    }
    return best_diffs;
}

static int
hamming_soft_fast(const mbo_soft_bit* in, char* out, int v) {
    int rc = check_soft_bits(in, 15);
    if (rc < 0) {
        return rc;
    }
    const uint16_t* rows = v ? ham_rows_7100 : ham_rows_std;
    uint32_t hard = 0;
    for (int i = 14; i >= 0; --i) {
        hard = (hard << 1) | (uint32_t)(in[i].bit & 1u);
    }
    int dummy;
    const uint32_t hard_fixed = ham_correct(hard, rows, &dummy);
    int tab[3][256];
    score_tables(in, 15, tab);
    int have = 0, best_score = 0x3fffffff, best_diffs = 0x3fffffff;
    uint32_t best = 0;
    for (uint32_t data = 0; data < 2048u; ++data) {
        const uint32_t cw = g_ham_cw[v][data];
        const uint32_t diff = cw ^ hard;
        const int score = tab[0][diff & 255u] + tab[1][diff >> 8];
        const int diffs = __builtin_popcount(diff);
        const int match = (cw == hard_fixed);
        const int best_match = have ? (best == hard_fixed) : 0;
        if (soft_better(have, score, best_score, match, best_match, diffs, best_diffs)) {
            best = cw;
            best_score = score;
            best_diffs = diffs;
            have = 1;
        }
    }
    for (int i = 0; i < 15; ++i) {
        out[i] = (char)((best >> i) & 1u);
    }
    return best_diffs;
}

typedef struct {
    int code, soft, fast, n, n_threads, tid;
    const uint8_t* in;
    uint8_t* out;
    int32_t* status;
} ecc_job_t;

static void*
ecc_worker(void* arg) {
    ecc_job_t* j = (ecc_job_t*)arg;
    const int len = j->code == 0 ? 23 : 15;
    for (int i = j->tid; i < j->n; i += j->n_threads) {
        char* o = (char*)(j->out + (size_t)i * len);
        int rc;
        if (j->soft) {
            const mbo_soft_bit* sb = (const mbo_soft_bit*)(j->in + (size_t)i * len * 2);
            if (j->fast) {
                rc = j->code == 0 ? golay_soft_fast(sb, o) : hamming_soft_fast(sb, o, j->code - 1);
            } else {
                rc = j->code == 0 ? mbo_golay2312_soft(sb, o) : mbo_hamming1511_soft(sb, o, j->code - 1);
            }
        } else {
            const char* b = (const char*)(j->in + (size_t)i * len);
            rc = j->code == 0 ? mbo_golay2312(b, o) : mbo_hamming1511(b, o, j->code - 1);
        }
        j->status[i] = rc;
    }
    return NULL;
}

void
mbo_ecc_blocks(int code, int soft, int fast, int n, const uint8_t* in, uint8_t* out, int32_t* status, int n_threads) {
    if (n_threads < 1) {
        n_threads = 1;
    }
    if (n_threads > 256) {
        n_threads = 256;
    }
    pthread_once(&g_cw_once, cw_tables_fill);
    ecc_job_t jobs[256];
    pthread_t th[256];
    for (int t = 0; t < n_threads; ++t) {
        ecc_job_t j = {code, soft, fast, n, n_threads, t, in, out, status};
        jobs[t] = j;
        if (n_threads > 1) {
            pthread_create(&th[t], NULL, ecc_worker, &jobs[t]);
        }
    }
    if (n_threads == 1) {
        ecc_worker(&jobs[0]);
    } else {
        for (int t = 0; t < n_threads; ++t) {
            pthread_join(th[t], NULL);
        }
    }
}
