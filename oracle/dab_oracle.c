/* oracle/dab_oracle.c -- TEST INFRASTRUCTURE, not product code.  See oracle/dab_oracle.h.
 *
 * Plain-C restatement of the reference DAB receive chain.  Paths cited are relative to
 * /root/reference/vendor/DAB-Radio/ ; VIT = vendor/viterbi_decoder/include/viterbi.
 * Build: oracle/Makefile target "port" (-O2, IEEE float, no contraction; fmaf() is written
 * explicitly where the pinned reference build (AVX2+FMA) fuses).
 */
#define _USE_MATH_DEFINES
#define _POSIX_C_SOURCE 200809L
#define _DEFAULT_SOURCE
#include "dab_oracle.h"
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif

/* =========================================================================================
 * Tables
 * ========================================================================================= */

/* Puncturing vectors in "bits kept per group of 4" form.  src/dab/constants/puncture_codes.h:42-67
 * (EN 300 401 table 13): PI_i keeps 8+i of 32 bits; extra bits go to groups 0,4,2,6,1,5,3,7. */
void dabo_pi_counts(int pi, uint8_t out8[8]) {
    static const int order[8] = {0, 4, 2, 6, 1, 5, 3, 7};
    const int base = 1 + (pi-1)/8;
    const int extra = (pi-1) % 8;
    for (int g = 0; g < 8; g++) out8[g] = (uint8_t)base;
    for (int k = 0; k <= extra; k++) out8[order[k]]++;
}

/* EEP profiles.  src/dab/constants/subchannel_protection_tables.h:121-154 ; msc_decoder.cpp:77-115 */
int dabo_eep_segments(int length, int level, int type_b, int seg_pi[3], int seg_bits[3]) {
    static const int A_mult[4] = {12, 8, 6, 4};
    static const int A_m[4][2] = {{6, 0}, {2, 4}, {6, 0}, {4, 2}};
    static const int A_b[4][2] = {{-3, 3}, {-3, 3}, {-3, 3}, {-3, 3}};
    static const int A_pi[4][2] = {{24, 23}, {14, 13}, {8, 7}, {3, 2}};
    static const int B_mult[4] = {27, 21, 18, 15};
    static const int B_pi[4][2] = {{10, 9}, {6, 5}, {4, 3}, {2, 1}};
    if (level < 0 || level > 3) return -1;
    int L1, L2, p1, p2;
    if (!type_b) {
        if (length == 8) {            /* the reference keys the 2-A n=1 special row on length only */
            L1 = 5; L2 = 1; p1 = 13; p2 = 12;
        } else {
            const int n = length / A_mult[level];
            L1 = A_m[level][0]*n + A_b[level][0];
            L2 = A_m[level][1]*n + A_b[level][1];
            p1 = A_pi[level][0]; p2 = A_pi[level][1];
        }
    } else {
        const int n = length / B_mult[level];
        L1 = 24*n - 3; L2 = 3;
        p1 = B_pi[level][0]; p2 = B_pi[level][1];
    }
    seg_pi[0] = p1; seg_bits[0] = 128*L1;
    seg_pi[1] = p2; seg_bits[1] = 128*L2;
    seg_pi[2] = 0;  seg_bits[2] = 24;
    return 3;
}

/* UEP profiles: L1..L4, PI1..PI4 per table index.  subchannel_protection_tables.h:21-86
 * (EN 300 401 tables 8 and 15).  Stored column-wise. */
static const uint8_t UEP_L[64][4] = {
    {3,4,17,0},{3,3,18,0},{3,4,14,3},{3,4,14,3},{3,5,13,3},{4,3,26,3},{3,4,26,3},{3,4,26,3},
    {3,4,26,3},{3,5,25,3},{6,10,23,3},{6,10,23,3},{6,12,21,3},{6,10,23,3},{6,9,31,2},{6,9,33,0},
    {6,12,27,3},{6,10,29,3},{6,11,28,3},{6,10,41,3},{6,10,41,3},{6,11,40,3},{6,10,41,3},{6,10,41,3},
    {7,9,53,3},{7,10,52,3},{6,12,51,3},{6,10,53,3},{6,13,50,3},{14,17,50,3},{11,21,49,3},{11,23,47,3},
    {11,21,49,3},{12,19,62,3},{11,21,61,3},{11,22,60,3},{11,21,61,3},{11,20,62,3},{11,19,87,3},{11,23,83,3},
    {11,24,82,3},{11,21,85,3},{11,22,84,3},{11,20,110,3},{11,22,108,3},{11,24,106,3},{11,20,110,3},{11,21,109,3},
    {12,22,131,3},{12,26,127,3},{11,20,134,3},{11,22,132,3},{11,24,130,3},{11,24,154,3},{11,24,154,3},{11,27,151,3},
    {11,22,156,3},{11,26,152,3},{11,26,200,3},{11,25,201,3},{11,26,200,3},{11,27,247,3},{11,24,250,3},{12,28,245,3},
};
static const uint8_t UEP_PI[64][4] = {
    {5,3,2,0},{11,6,5,0},{15,9,6,8},{22,13,8,13},{24,17,12,17},{5,4,2,3},{9,6,4,6},{15,10,6,9},
    {24,14,8,15},{24,18,13,18},{5,4,2,3},{9,6,4,5},{16,7,6,9},{23,13,8,13},{5,3,2,3},{11,6,5,0},
    {16,8,6,9},{23,13,8,13},{24,18,12,18},{6,3,2,3},{11,6,5,6},{16,8,6,7},{23,13,8,13},{24,17,12,18},
    {5,4,2,4},{9,6,4,6},{16,9,6,10},{22,12,9,12},{24,18,13,19},{5,4,2,5},{9,6,4,8},{16,8,6,9},
    {23,12,9,14},{5,3,2,4},{11,6,5,7},{16,9,6,10},{22,12,9,14},{24,17,13,19},{5,4,2,4},{11,6,5,9},
    {16,8,6,11},{22,11,9,13},{24,18,12,19},{6,4,2,5},{10,6,4,9},{16,10,6,11},{22,13,9,13},{24,20,13,24},
    {8,6,2,6},{12,8,4,11},{16,10,7,9},{24,16,10,15},{24,20,12,20},{6,5,2,5},{12,9,5,10},{16,10,7,10},
    {24,14,10,13},{24,19,14,18},{8,5,2,6},{13,9,5,10},{24,17,9,17},{8,6,2,7},{16,9,7,10},{24,20,14,23},
};

int dabo_uep_segments(int index, int seg_pi[5], int seg_bits[5]) {
    if (index < 0 || index >= 64) return -1;
    int n = 0;
    for (int i = 0; i < 4; i++) {
        if (UEP_L[index][i] == 0) continue;       /* update() with 0 requested symbols is a no-op */
        seg_pi[n] = UEP_PI[index][i];
        seg_bits[n] = 128*UEP_L[index][i];
        n++;
    }
    seg_pi[n] = 0; seg_bits[n] = 24; n++;
    return n;
}

/* src/ofdm/dab_ofdm_params_ref.cpp:10-58 */
int dabo_ofdm_params(int mode, int out6[6]) {
    static const int T[4][6] = {
        {76, 2552, 2656, 504, 2048, 1536},
        {76,  638,  664, 126,  512,  384},
        {153, 319,  345,  63,  256,  192},
        {76, 1276, 1328, 252, 1024,  768},
    };
    if (mode < 1 || mode > 4) return -1;
    memcpy(out6, T[mode-1], sizeof(T[0]));
    return 0;
}

/* src/ofdm/dab_mapper_ref.cpp:10-50 (EN 300 401 clause 14.6.1) */
int dabo_carrier_map(int nb_fft, int nb_carriers, int* out) {
    const int dc = nb_fft/2, lo = dc - nb_carriers/2, hi = dc + nb_carriers/2;
    int v = 0, n = 0;
    for (int i = 0; i < nb_fft; i++) {
        if (i > 0) v = (13*v + nb_fft/4 - 1) % nb_fft;
        if (v < lo || v > hi || v == dc) continue;
        out[n++] = (v < dc) ? (v - lo) : (v - lo - 1);
    }
    return n;
}

/* src/ofdm/dab_prs_ref.cpp:24-194 (EN 300 401 clause 14.3.2, tables 23/24) */
static const uint8_t PRS_H[4][32] = {
    {0,2,0,0,0,0,1,1,2,0,0,0,2,2,1,1,0,2,0,0,0,0,1,1,2,0,0,0,2,2,1,1},
    {0,3,2,3,0,1,3,0,2,1,2,3,2,3,3,0,0,3,2,3,0,1,3,0,2,1,2,3,2,3,3,0},
    {0,0,0,2,0,2,1,3,2,2,0,2,2,0,1,3,0,0,0,2,0,2,1,3,2,2,0,2,2,0,1,3},
    {0,1,2,1,0,3,3,2,2,3,2,1,2,1,3,2,0,1,2,1,0,3,3,2,2,3,2,1,2,1,3,2},
};
/* (i<<2)|n for each block of 32 carriers from -K/2 upwards (DC skipped) */
static const uint8_t PRS_IN_1[48] = {
    0x1,0x6,0x8,0xd,0x3,0x6,0xa,0xf,0x2,0x5,0xa,0xf,0x1,0x6,0xb,0xf,0x2,0x6,0xa,0xd,0x1,0x7,0x9,0xe,
    0x3,0xd,0x9,0x5,0x2,0xe,0x9,0x4,0x2,0xe,0xb,0x7,0x0,0xe,0x9,0x7,0x3,0xf,0xb,0x4,0x3,0xc,0x9,0x5};
static const uint8_t PRS_IN_2[12] = {0x2,0x7,0xa,0xe,0x1,0x6, 0x8,0x6,0x2,0xd,0x8,0x7};
static const uint8_t PRS_IN_3[6]  = {0x2,0x7,0x8, 0xe,0xa,0x6};
static const uint8_t PRS_IN_4[24] = {
    0x0,0x5,0x9,0xe,0x2,0x6,0x8,0xf,0x3,0x5,0xb,0xe,
    0x0,0xd,0x8,0x6,0x0,0xd,0xa,0x6,0x2,0xd,0xb,0x4};

int dabo_prs_fft(int mode, float* out, int nb_fft) {
    int P[6];
    if (dabo_ofdm_params(mode, P) != 0) return -1;
    const int K = P[5];
    const uint8_t* tab = (mode == 1) ? PRS_IN_1 : (mode == 2) ? PRS_IN_2 : (mode == 3) ? PRS_IN_3 : PRS_IN_4;
    if (nb_fft < K+1) return -1;
    memset(out, 0, sizeof(float)*2*(size_t)nb_fft);
    for (int slot = 0; slot < K; slot++) {
        const int k = (slot < K/2) ? (slot - K/2) : (slot - K/2 + 1);
        const int blk = slot/32, j = slot%32;
        const int i = tab[blk] >> 2, n = tab[blk] & 3;
        const float phi = (float)M_PI / 2.0f * (float)(PRS_H[i][j] + n);
        const int bin = (k < 0) ? (nb_fft + k) : k;
        out[2*bin+0] = cosf(phi);
        out[2*bin+1] = sinf(phi);
    }
    return 0;
}

/* =========================================================================================
 * Viterbi K=7 R=1/4: scalar statement of the AVX2 u16 decoder
 *   VIT/x86/viterbi_decoder_avx_u16.h:47-170 (update/bfly/renormalise)
 *   VIT/viterbi_branch_table.h:45-55, VIT/viterbi_decoder_core.h:180-236 (reset, chainback)
 *   src/dab/algorithms/dab_viterbi_decoder.cpp:18-41 (polynomials, config), 131-181 (depuncture)
 * ========================================================================================= */
#define VIT_STATES 64
#define VIT_MAX_ERROR 1016u          /* (127 - -127) * 4 */
#define VIT_NONSTART  5080u          /* 5 * max_error */
#define VIT_RENORM    60455u         /* 65535 - 5080 */
static const uint8_t VIT_POLY[4] = {109, 79, 83, 109};
static int16_t VIT_BT[4][32];
static int vit_bt_ready = 0;

static int parity8(unsigned v) { v ^= v >> 4; v ^= v >> 2; v ^= v >> 1; return (int)(v & 1u); }

static void vit_init_tables(void) {
    if (vit_bt_ready) return;
    for (int s = 0; s < 32; s++)
        for (int r = 0; r < 4; r++)
            VIT_BT[r][s] = parity8(((unsigned)s << 1) & VIT_POLY[r]) ? 127 : -127;
    vit_bt_ready = 1;
}

static inline uint16_t addsat_u16(uint16_t a, uint16_t b) { const uint32_t s = (uint32_t)a + b; return (uint16_t)(s > 65535u ? 65535u : s); }

typedef struct {
    uint16_t metric[2][VIT_STATES];
    int cur;
    uint64_t* decisions;
    size_t cap_steps;
    size_t step;
    uint64_t accumulated_error;
} vit_t;

static void vit_reset(vit_t* v) {
    v->cur = 0; v->step = 0; v->accumulated_error = 0;
    for (int i = 0; i < VIT_STATES; i++) v->metric[0][i] = VIT_NONSTART;
    v->metric[0][0] = 0;
}

static void vit_update(vit_t* v, const int16_t* sym, size_t n_sym) {
    for (size_t k = 0; k < n_sym; k += 4) {
        const uint16_t* old = v->metric[v->cur];
        uint16_t* nw = v->metric[1 - v->cur];
        uint64_t dec = 0;
        for (int s = 0; s < 32; s++) {
            uint32_t e = 0;
            for (int r = 0; r < 4; r++) {
                int d = (int)VIT_BT[r][s] - (int)sym[k + (size_t)r];
                if (d > 32767) d = 32767;
                if (d < -32768) d = -32768;
                e += (uint32_t)(d < 0 ? -d : d);
            }
            if (e > 65535u) e = 65535u;
            const uint16_t err = (uint16_t)e;
            const uint16_t inv = (uint16_t)(VIT_MAX_ERROR > e ? VIT_MAX_ERROR - e : 0u);
            const uint16_t n00 = addsat_u16(old[s], err);
            const uint16_t n10 = addsat_u16(old[s + 32], inv);
            const uint16_t n01 = addsat_u16(old[s], inv);
            const uint16_t n11 = addsat_u16(old[s + 32], err);
            const uint16_t m0 = n00 < n10 ? n00 : n10;
            const uint16_t m1 = n01 < n11 ? n01 : n11;
            nw[2*s] = m0;
            nw[2*s + 1] = m1;
            if (m0 == n10) dec |= (uint64_t)1 << (2*s);        /* tie => 1 */
            if (m1 == n11) dec |= (uint64_t)1 << (2*s + 1);
        }
        v->decisions[v->step] = dec;
        if (nw[0] >= VIT_RENORM) {
            uint16_t mn = nw[0];
            for (int i = 1; i < VIT_STATES; i++) if (nw[i] < mn) mn = nw[i];
            for (int i = 0; i < VIT_STATES; i++) nw[i] = (uint16_t)(nw[i] - mn);
            v->accumulated_error += mn;
        }
        v->cur = 1 - v->cur;
        v->step++;
    }
}

static void vit_chainback(const vit_t* v, uint8_t* out, size_t total_bits) {
    unsigned reg = 0;   /* 8-bit window, state = reg >> 2 (end state 0) */
    for (size_t i = 0; i < total_bits; i++) {
        const size_t j = total_bits - 1 - i;
        const uint64_t d = v->decisions[j + 6];
        const unsigned state = reg >> 2;
        const unsigned bit = (unsigned)((d >> state) & 1u);
        reg = (reg >> 1) | (bit << 7);
        out[j/8] = (uint8_t)reg;
    }
}

/* depuncture_symbols, dab_viterbi_decoder.cpp:131-181 */
static int depuncture(const int8_t* in, int n_in, const uint8_t* code, int code_len, int n_out, int16_t* out, int* consumed) {
    int ip = 0, ic = 0, io = 0;
    while (io < n_out) {
        const int keep = code[ic];
        if (n_in - ip < keep) { *consumed = 0; return 0; }   /* reference returns zeros here */
        for (int i = 0; i < keep; i++) out[io++] = (int16_t)in[ip++];
        for (int i = keep; i < 4; i++) out[io++] = 0;
        ic = (ic + 1) % code_len;
    }
    *consumed = ip;
    return io;
}

static const uint8_t PI_X_CODE[6] = {2, 2, 2, 2, 2, 2};

int dabo_vit_decode(const int8_t* soft, int n_soft, const int* seg_pi, const int* seg_bits, int n_seg,
                    uint8_t* out_bytes, int n_out_bytes, uint64_t* path_error) {
    vit_init_tables();
    int total_steps = 0, max_seg = 0;
    for (int i = 0; i < n_seg; i++) { total_steps += seg_bits[i]/4; if (seg_bits[i] > max_seg) max_seg = seg_bits[i]; }
    if (n_out_bytes*8 + 6 > total_steps) return -1;
    vit_t v;
    v.decisions = (uint64_t*)malloc(sizeof(uint64_t)*(size_t)(total_steps > 0 ? total_steps : 1));
    v.cap_steps = (size_t)total_steps;
    int16_t* dep = (int16_t*)malloc(sizeof(int16_t)*(size_t)(max_seg > 0 ? max_seg : 4));
    vit_reset(&v);
    int consumed_total = 0;
    for (int i = 0; i < n_seg; i++) {
        uint8_t code[8];
        const uint8_t* c; int clen;
        if (seg_pi[i] == 0) { c = PI_X_CODE; clen = 6; } else { dabo_pi_counts(seg_pi[i], code); c = code; clen = 8; }
        int consumed = 0;
        const int n = depuncture(soft + consumed_total, n_soft - consumed_total, c, clen, seg_bits[i], dep, &consumed);
        vit_update(&v, dep, (size_t)n);
        consumed_total += consumed;
    }
    vit_chainback(&v, out_bytes, (size_t)n_out_bytes*8u);
    if (path_error) *path_error = v.accumulated_error + v.metric[v.cur][0];
    free(dep); free(v.decisions);
    return consumed_total;
}

/* =========================================================================================
 * Energy dispersal, CRC.  additive_scrambler.h:10-36 ; crc.h:11-68
 * ========================================================================================= */
void dabo_scrambler_bytes(uint8_t* out, int n) {
    uint16_t reg = 0xFFFF;
    for (int k = 0; k < n; k++) {
        uint8_t b = 0;
        for (int i = 0; i < 8; i++) {
            const uint8_t v = (uint8_t)(((reg >> 8) ^ (reg >> 4)) & 1u);
            b |= (uint8_t)(v << (7 - i));
            reg = (uint16_t)((reg << 1) | v);
        }
        out[k] = b;
    }
}

uint16_t dabo_crc16(const uint8_t* data, int n, uint16_t poly, uint16_t init, uint16_t xorout) {
    uint16_t crc = init;
    for (int i = 0; i < n; i++) {
        crc ^= (uint16_t)(data[i] << 8);
        for (int b = 0; b < 8; b++) crc = (crc & 0x8000u) ? (uint16_t)((crc << 1) ^ poly) : (uint16_t)(crc << 1);
    }
    return (uint16_t)(crc ^ xorout);
}

/* =========================================================================================
 * FIC.  src/dab/fic/fic_decoder.cpp:53-117
 * ========================================================================================= */
int dabo_fic_decode_group(const int8_t* bits, uint8_t out96[96], int crc_ok[3]) {
    static const int pi[3] = {16, 15, 0};
    static const int nb[3] = {128*21, 128*3, 24};
    uint8_t prbs[96];
    if (dabo_vit_decode(bits, 2304, pi, nb, 3, out96, 96, NULL) != 2304) return -1;
    dabo_scrambler_bytes(prbs, 96);
    for (int i = 0; i < 96; i++) out96[i] ^= prbs[i];
    int n_ok = 0;
    for (int f = 0; f < 3; f++) {
        const uint8_t* fib = out96 + 32*f;
        const uint16_t rx = (uint16_t)((fib[30] << 8) | fib[31]);
        crc_ok[f] = (dabo_crc16(fib, 30, 0x1021, 0xFFFF, 0xFFFF) == rx);
        n_ok += crc_ok[f];
    }
    return n_ok;
}

/* =========================================================================================
 * MSC sub-channel: time de-interleave + EEP/UEP decode.
 *   src/dab/msc/cif_deinterleaver.cpp:8-71 ; src/dab/msc/msc_decoder.cpp:46-154
 * ========================================================================================= */
static const int TI_OFFSETS[16] = {0,8,4,12, 2,10,6,14, 1,9,5,13, 3,11,7,15};

struct dabo_msc {
    int start_address, length, is_uep, uep_index, eep_level, eep_type_b;
    int nb_bits;
    int8_t* ring;      /* 16 x nb_bits */
    int curr_frame, total_stored;
    int8_t* deint;
    uint8_t* prbs;
};

dabo_msc* dabo_msc_create(int start_address, int length, int is_uep, int uep_index, int eep_level, int eep_type_b) {
    dabo_msc* m = (dabo_msc*)calloc(1, sizeof(*m));
    m->start_address = start_address; m->length = length; m->is_uep = is_uep; m->uep_index = uep_index;
    m->eep_level = eep_level; m->eep_type_b = eep_type_b;
    m->nb_bits = length*64;
    m->ring = (int8_t*)calloc((size_t)m->nb_bits*16u, 1);
    m->deint = (int8_t*)calloc((size_t)m->nb_bits, 1);
    m->prbs = (uint8_t*)malloc((size_t)length*8u);
    dabo_scrambler_bytes(m->prbs, length*8);
    return m;
}
void dabo_msc_destroy(dabo_msc* m) { if (!m) return; free(m->ring); free(m->deint); free(m->prbs); free(m); }

int dabo_msc_decode_cif(dabo_msc* m, const int8_t* cif, int n_bits, uint8_t* out, int out_cap) {
    const int start = m->start_address*64;
    if (start + m->nb_bits > n_bits) return 0;
    memcpy(m->ring + (size_t)m->curr_frame*(size_t)m->nb_bits, cif + start, (size_t)m->nb_bits);
    m->curr_frame = (m->curr_frame + 1) % 16;
    if (m->total_stored < 16) m->total_stored++;
    if (m->total_stored < 16) return 0;
    for (int i = 0; i < m->nb_bits; i++) {
        const int age = 15 - TI_OFFSETS[i % 16];                 /* 0 = newest */
        const int row = ((m->curr_frame - 1) - age + 32) % 16;
        m->deint[i] = m->ring[(size_t)row*(size_t)m->nb_bits + (size_t)i];
    }
    int pi[5], nb[5], nseg;
    if (m->is_uep) nseg = dabo_uep_segments(m->uep_index, pi, nb);
    else           nseg = dabo_eep_segments(m->length, m->eep_level, m->eep_type_b, pi, nb);
    if (nseg < 0) return 0;
    /* A segment whose punctured symbols no longer fit the sub-channel decodes nothing and consumes nothing: depuncture_symbols
     * returns an all-zero result when a block runs out of input (dab_viterbi_decoder.cpp:157-161) and DecodeUEP / DecodeEEP go on
     * with the next update() (msc_decoder.cpp:86-96, 128-139).  Hits UEP row 34, which the reference's table lists with 64 CU. */
    {
        int remaining = m->nb_bits, k = 0;
        for (int i = 0; i < nseg; i++) {
            int need = 0;
            uint8_t cnt[8] = {2, 2, 2, 2, 2, 2, 2, 2};            /* PI_X keeps 2 of every 4 mother bits */
            if (pi[i] != 0) dabo_pi_counts(pi[i], cnt);
            for (int g = 0; g < nb[i]/4; g++) need += cnt[g % 8];
            if (need > remaining) continue;
            remaining -= need;
            pi[k] = pi[i]; nb[k] = nb[i]; k++;
        }
        nseg = k;
    }
    int steps = 0;
    for (int i = 0; i < nseg; i++) steps += nb[i]/4;
    const int n_bytes = (steps - 6)/8;
    if (n_bytes > out_cap) return -n_bytes;
    dabo_vit_decode(m->deint, m->nb_bits, pi, nb, nseg, out, n_bytes, NULL);
    for (int i = 0; i < n_bytes; i++) out[i] ^= m->prbs[i];
    return n_bytes;
}

/* =========================================================================================
 * Reed-Solomon over GF(2^8)/0x11D, fcr 0, prim 1 (Phil Karn's decode_rs algorithm).
 *   src/dab/algorithms/reed_solomon_decoder.cpp:70-178 (field tables), 192-477 (decode)
 * ========================================================================================= */
static uint8_t GF_EXP[256], GF_LOG[256];
static int gf_ready = 0;
static void gf_init(void) {
    if (gf_ready) return;
    int sr = 1;
    GF_LOG[0] = 255; GF_EXP[255] = 0;
    for (int i = 0; i < 255; i++) {
        GF_LOG[sr] = (uint8_t)i; GF_EXP[i] = (uint8_t)sr;
        sr <<= 1; if (sr & 0x100) sr ^= 0x11D; sr &= 255;
    }
    gf_ready = 1;
}
static inline int mod255(int x) { while (x >= 255) { x -= 255; x = (x >> 8) + (x & 255); } return x; }
static inline uint8_t gf_mul(uint8_t a, uint8_t b) { return (a && b) ? GF_EXP[mod255(GF_LOG[a] + GF_LOG[b])] : 0; }

int dabo_rs_decode(int nroots, int pad, uint8_t* data, int* eras_pos) {
    gf_init();
    if (nroots < 1 || nroots > 32) return -1;
    const int n = 255 - pad;
    uint8_t S[32], lambda[33], b[33], t[33], omega[33], root[32], loc[32];
    /* syndromes S_i = data(alpha^i), Horner with data[0] the highest-degree coefficient */
    int nonzero = 0;
    for (int i = 0; i < nroots; i++) {
        uint8_t s = data[0];
        for (int j = 1; j < n; j++) s = (uint8_t)(data[j] ^ (s ? GF_EXP[mod255(GF_LOG[s] + i)] : 0));
        S[i] = s; nonzero |= s;
    }
    int count = 0;
    if (!nonzero) goto finish;
    /* Berlekamp-Massey */
    memset(lambda, 0, sizeof(lambda)); memset(b, 0, sizeof(b));
    lambda[0] = 1; b[0] = 1;
    int el = 0;
    for (int r = 1; r <= nroots; r++) {
        uint8_t discr = 0;
        for (int i = 0; i < r; i++) discr ^= gf_mul(lambda[i], S[r-i-1]);
        if (discr == 0) {
            memmove(&b[1], b, (size_t)nroots); b[0] = 0;
        } else {
            t[0] = lambda[0];
            for (int i = 0; i < nroots; i++) t[i+1] = (uint8_t)(lambda[i+1] ^ gf_mul(discr, b[i]));
            if (2*el <= r - 1) {
                el = r - el;
                const int ld = GF_LOG[discr];
                for (int i = 0; i <= nroots; i++) b[i] = lambda[i] ? GF_EXP[mod255(GF_LOG[lambda[i]] - ld + 255)] : 0;
            } else {
                memmove(&b[1], b, (size_t)nroots); b[0] = 0;
            }
            memcpy(lambda, t, (size_t)nroots + 1);
        }
    }
    int deg_lambda = 0;
    for (int i = 0; i <= nroots; i++) if (lambda[i]) deg_lambda = i;
    /* Chien search: i = 1..255, location k = i-1 (prim = 1 => iprim = 1) */
    for (int i = 1; i <= 255; i++) {
        uint8_t q = 1;
        for (int j = deg_lambda; j > 0; j--) if (lambda[j]) q ^= GF_EXP[mod255(GF_LOG[lambda[j]] + (i*j) % 255)];
        if (q != 0) continue;
        root[count] = (uint8_t)i; loc[count] = (uint8_t)(i - 1);
        if (++count == deg_lambda) break;
    }
    if (deg_lambda != count) { count = -1; goto finish; }
    /* omega = S * lambda mod x^nroots */
    const int deg_omega = deg_lambda - 1;
    for (int i = 0; i <= deg_omega; i++) {
        uint8_t tmp = 0;
        for (int j = i; j >= 0; j--) tmp ^= gf_mul(S[i-j], lambda[j]);
        omega[i] = tmp;
    }
    /* Forney, fcr = 0 */
    for (int j = count-1; j >= 0; j--) {
        uint8_t num1 = 0, den = 0;
        for (int i = deg_omega; i >= 0; i--) if (omega[i]) num1 ^= GF_EXP[mod255(GF_LOG[omega[i]] + (i*root[j]) % 255)];
        const uint8_t num2 = GF_EXP[mod255(255 - root[j])];
        const int top = (deg_lambda < nroots-1 ? deg_lambda : nroots-1) & ~1;
        for (int i = top; i >= 0; i -= 2) if (lambda[i+1]) den ^= GF_EXP[mod255(GF_LOG[lambda[i+1]] + (i*root[j]) % 255)];
        if (num1 != 0 && loc[j] >= pad) {
            data[loc[j] - pad] ^= GF_EXP[mod255(GF_LOG[num1] + GF_LOG[num2] + 255 - GF_LOG[den])];
        }
    }
finish:
    if (eras_pos) for (int i = 0; i < count; i++) eras_pos[i] = loc[i];
    return count;
}

/* =========================================================================================
 * DAB+ superframe processor.  src/dab/audio/aac_frame_processor.cpp:126-362
 * ========================================================================================= */
enum { EV_FIRECODE_ERROR = 1, EV_RS_ERROR = 2, EV_HEADER = 3, EV_AU_CRC_ERROR = 4, EV_AU = 5 };
struct dabo_aac {
    int state_collect;       /* 0 WAIT_FRAME_START, 1 COLLECT_FRAMES */
    int curr_frame, prev_nb, synced, desync;
    uint8_t* sf; int sf_cap;
    uint8_t* log; int log_len, log_cap;
};
dabo_aac* dabo_aac_create(void) { return (dabo_aac*)calloc(1, sizeof(dabo_aac)); }
void dabo_aac_destroy(dabo_aac* a) { if (!a) return; free(a->sf); free(a->log); free(a); }

static void aac_ev(dabo_aac* a, int type, int x, int y, int z, int w, const uint8_t* payload, int nbytes) {
    const int pad = (nbytes + 3) & ~3;
    if (a->log_len + 24 + pad > a->log_cap) {
        a->log_cap = (a->log_len + 24 + pad)*2;
        a->log = (uint8_t*)realloc(a->log, (size_t)a->log_cap);
    }
    int32_t hdr[6] = {type, x, y, z, w, nbytes};
    memcpy(a->log + a->log_len, hdr, 24);
    memset(a->log + a->log_len + 24, 0, (size_t)pad);
    if (nbytes > 0) memcpy(a->log + a->log_len + 24, payload, (size_t)nbytes);
    a->log_len += 24 + pad;
}

static int aac_firecode_ok(dabo_aac* a, const uint8_t* buf) {
    const uint16_t rx = (uint16_t)((buf[0] << 8) | buf[1]);
    const uint16_t pred = dabo_crc16(buf + 2, 9, 0x782F, 0, 0);
    if (rx != pred) aac_ev(a, EV_FIRECODE_ERROR, a->curr_frame, rx, pred, 0, NULL, 0);
    return rx == pred;
}

/* read_au_start, aac_frame_processor.cpp:30-72: n 12-bit values, MSB first; returns bytes consumed */
static int read_au_start(const uint8_t* buf, uint16_t* data, int n) {
    int bitpos = 0;
    for (int i = 0; i < n; i++) {
        unsigned v = 0;
        for (int k = 0; k < 12; k++, bitpos++) v = (v << 1) | ((buf[bitpos >> 3] >> (7 - (bitpos & 7))) & 1u);
        data[i] = (uint16_t)v;
    }
    return (bitpos + 7) >> 3;
}

static void aac_process_superframe(dabo_aac* a, int nb_frame_bytes) {
    const int total = nb_frame_bytes*5;
    const int N = total/120;
    uint8_t cw[120]; int pos[10];
    for (int i = 0; i < N; i++) {
        for (int j = 0; j < 120; j++) cw[j] = a->sf[i + j*N];
        const int cnt = dabo_rs_decode(10, 135, cw, pos);
        if (cnt < 0) { aac_ev(a, EV_RS_ERROR, i, N, 0, 0, NULL, 0); a->desync++; return; }
        for (int j = 0; j < cnt; j++) {
            const int k = pos[j] - 135;
            if (k < 0) continue;
            a->sf[i + k*N] = cw[k];
        }
    }
    if (!aac_firecode_ok(a, a->sf)) { a->desync++; return; }
    a->desync = 0; a->synced = 1;
    const uint8_t d = a->sf[2];
    const int dac_rate = (d >> 6) & 1, sbr = (d >> 5) & 1, ch = (d >> 4) & 1, ps = (d >> 3) & 1, mpeg = d & 7;
    const int surround = (mpeg == 0) ? 0 : (mpeg == 1) ? 1 : (mpeg == 2) ? 2 : (mpeg == 7) ? 3 : 4;
    aac_ev(a, EV_HEADER, dac_rate ? 48000 : 32000, (ps ? 1 : 0) | (sbr ? 2 : 0) | (ch ? 4 : 0), surround, 0, NULL, 0);
    int num_aus = 0;
    if (!dac_rate && sbr) num_aus = 2;
    if (dac_rate && sbr) num_aus = 3;
    if (!dac_rate && !sbr) num_aus = 4;
    if (dac_rate && !sbr) num_aus = 6;
    uint16_t au_start[7] = {0};
    const int nb_tbl = read_au_start(a->sf + 3, &au_start[1], num_aus - 1);
    au_start[num_aus] = (uint16_t)(110*N);
    au_start[0] = (uint16_t)(3 + nb_tbl);
    for (int i = 0; i < num_aus; i++) {
        const int nb_au = (int)au_start[i+1] - (int)au_start[i];
        const int nb_data = nb_au - 2;
        if (nb_data < 0 || au_start[i+1] >= total) return;
        const uint8_t* au = a->sf + au_start[i];
        const uint16_t rx = (uint16_t)((au[nb_data] << 8) | au[nb_data+1]);
        const uint16_t pred = dabo_crc16(au, nb_data, 0x1021, 0xFFFF, 0xFFFF);
        if (rx != pred) { aac_ev(a, EV_AU_CRC_ERROR, i, num_aus, rx, pred, NULL, 0); continue; }
        aac_ev(a, EV_AU, i, num_aus, 0, 0, au, nb_data);
    }
}

int dabo_aac_process(dabo_aac* a, const uint8_t* frame, int n, uint8_t* log_out, int log_cap) {
    a->log_len = 0;
    if (n == 0 || n < 11) return 0;
    if (a->prev_nb != n) {
        a->prev_nb = n;
        if (a->sf_cap < 5*n) { a->sf = (uint8_t*)realloc(a->sf, (size_t)5*(size_t)n); a->sf_cap = 5*n; }
        a->curr_frame = 0; a->state_collect = 0;
    }
    if (a->desync >= 10) { a->desync = 0; a->synced = 0; }
    if (a->synced) a->state_collect = 1;
    if (!a->state_collect) {
        if (!aac_firecode_ok(a, frame)) goto done;
        a->state_collect = 1;
    }
    memcpy(a->sf + (size_t)a->curr_frame*(size_t)n, frame, (size_t)n);
    a->curr_frame++;
    if (a->curr_frame == 5) {
        aac_process_superframe(a, n);
        a->state_collect = 0; a->curr_frame = 0;
    }
done:
    if (a->log_len > 0 && a->log_len <= log_cap) memcpy(log_out, a->log, (size_t)a->log_len);
    return a->log_len;
}

/* =========================================================================================
 * OFDM demodulator, canonical serialised order (SURVEY.md appendix C).
 *   src/ofdm/ofdm_demodulator.cpp:235-950, src/ofdm/dsp/apply_pll.cpp:82-116,
 *   src/ofdm/dsp/chebyshev_sine.h:79-105, src/ofdm/dsp/complex_conj_mul_sum.cpp:65-99,
 *   src/ofdm/circular_buffer.h, reconstruction_buffer.h, ofdm_frame_buffer.h
 * ========================================================================================= */
typedef struct { float re, im; } cf;

/* iterative radix-2 DIT, unnormalised, twiddles rounded from double */
typedef struct { int n; cf* tw; int* rev; } fftplan;
static fftplan* fft_make(int n) {
    fftplan* p = (fftplan*)malloc(sizeof(*p));
    p->n = n; p->tw = (cf*)malloc(sizeof(cf)*(size_t)n/2); p->rev = (int*)malloc(sizeof(int)*(size_t)n);
    int bits = 0; while ((1 << bits) < n) bits++;
    for (int i = 0; i < n; i++) { int r = 0; for (int b = 0; b < bits; b++) if (i & (1 << b)) r |= 1 << (bits-1-b); p->rev[i] = r; }
    for (int k = 0; k < n/2; k++) { const double a = -2.0*M_PI*(double)k/(double)n; p->tw[k].re = (float)cos(a); p->tw[k].im = (float)sin(a); }
    return p;
}
static void fft_free(fftplan* p) { if (!p) return; free(p->tw); free(p->rev); free(p); }
static void fft_exec(const fftplan* p, const cf* in, cf* out, int inverse) {
    const int n = p->n;
    if (in == out) {
        for (int i = 0; i < n; i++) { const int r = p->rev[i]; if (r > i) { cf t = out[i]; out[i] = out[r]; out[r] = t; } }
    } else {
        for (int i = 0; i < n; i++) out[p->rev[i]] = in[i];
    }
    for (int len = 2; len <= n; len <<= 1) {
        const int half = len/2, step = n/len;
        for (int i = 0; i < n; i += len) {
            for (int k = 0; k < half; k++) {
                cf w = p->tw[k*step];
                if (inverse) w.im = -w.im;
                const cf a = out[i+k], b = out[i+k+half];
                const float tr = b.re*w.re - b.im*w.im, ti = b.re*w.im + b.im*w.re;
                out[i+k].re = a.re + tr; out[i+k].im = a.im + ti;
                out[i+k+half].re = a.re - tr; out[i+k+half].im = a.im - ti;
            }
        }
    }
}
void dabo_fft(float* data, int n, int inverse) {
    fftplan* p = fft_make(n);
    fft_exec(p, (const cf*)data, (cf*)data, inverse);
    fft_free(p);
}

enum { ST_FINDING_NULL = 0, ST_READING_NULL_PRS = 1, ST_COARSE = 2, ST_FINE_TIME = 3, ST_READING_SYMBOLS = 4 };

typedef struct frame_node { struct frame_node* next; float coarse, fine; int time_offset; int8_t bits[]; } frame_node;

struct dabo_ofdm {
    int mode, L, Tsym, Tnull, CP, N, K;
    /* config, ofdm_demodulator.h:24-45 */
    float l1_beta; int l1_nb_samples, l1_decimate;
    float thresh_null_start, thresh_null_end;
    float fine_beta; int coarse_enabled; float max_coarse_norm, coarse_slow_beta, impulse_thresh_db, impulse_dist_prob;
    /* state */
    int state, frames_read, frames_desync, coarse_found, fine_time_offset, null_start_found, null_end_found;
    float coarse, fine, l1_avg;
    /* buffers */
    cf* null_ring; size_t ring_index, ring_len;
    cf* corr; size_t corr_len;
    cf* frame; size_t frame_fill, frame_cap;
    cf *prs_fft_conj, *prs_time_ref, *fftbuf, *ifftbuf, *spectra;
    float *impulse, *freq_resp, *phase_err;
    int* cmap;
    fftplan* plan;
    cf* scratch; size_t scratch_cap;
    int keep;
    frame_node *q_head, *q_tail;
};

static float cabs_f(cf v) { return sqrtf(v.re*v.re + v.im*v.im); }

/* chebyshev_sine.h:13-20, evaluated as the AVX+FMA build does: ((x*g(z)) * (z-0.25)) */
static inline float cheb_sin(float x) {
    const float z = x*x;
    float b = 3.20396066f;
    b = fmaf(b, z, -14.07150173f);
    b = fmaf(b, z, 38.50016403f);
    b = fmaf(b, z, -67.07687378f);
    b = fmaf(b, z, 64.83583069f);
    b = fmaf(b, z, -25.13274193f);
    return (x*b)*(z + -0.25f);
}

/* apply_pll_avx, dsp/apply_pll.cpp:82-116 (vector body; the scalar tail of lengths not divisible by 4
 * differs only in association, which is inside the soft-bit tolerance) */
static void apply_pll(const cf* x, cf* y, size_t n, float f, float dt0) {
    float off_s[4], off_c[4];
    for (int k = 0; k < 4; k++) { const float d = (float)k*f; off_s[k] = d; off_c[k] = d + 0.25f; }
    for (size_t i = 0; i < n; i++) {
        const size_t i4 = i & ~(size_t)3; const int k = (int)(i & 3);
        const float base = fmaf((float)i4, f, dt0);
        float ts = base + off_s[k], tc = base + off_c[k];
        ts = ts - rintf(ts); tc = tc - rintf(tc);
        const float s = cheb_sin(ts), c = cheb_sin(tc);
        const cf v = x[i];
        y[i].re = fmaf(c, v.re, -(s*v.im));
        y[i].im = fmaf(c, v.im,  (s*v.re));
    }
}

/* complex_conj_mul_sum_avx: sum x0[i]*conj(x1[i]) with 4 interleaved partial sums */
static cf conj_mul_sum(const cf* x0, const cf* x1, size_t n) {
    float pr[4] = {0,0,0,0}, pi[4] = {0,0,0,0};
    const size_t nv = n & ~(size_t)3;
    for (size_t i = 0; i < nv; i++) {
        const int k = (int)(i & 3);
        pr[k] += fmaf(x0[i].im, x1[i].im, x0[i].re*x1[i].re);
        pi[k] += fmaf(x0[i].im, x1[i].re, -(x0[i].re*x1[i].im));
    }
    cf y; y.re = (pr[0]+pr[2]) + (pr[1]+pr[3]); y.im = (pi[0]+pi[2]) + (pi[1]+pi[3]);
    for (size_t i = nv; i < n; i++) { y.re += x0[i].re*x1[i].re + x0[i].im*x1[i].im; y.im += x0[i].im*x1[i].re - x0[i].re*x1[i].im; }
    return y;
}

static float l1_average(const cf* b, size_t n) {
    float s = 0.0f;
    for (size_t i = 0; i < n; i++) s += fabsf(b[i].re) + fabsf(b[i].im);
    return s/(float)n;
}

static void update_fine(dabo_ofdm* d, float delta) {      /* ofdm_demodulator.cpp:829-840 */
    const float wrap = 0.5f*(1.0f/(float)d->N)*1.01f;
    d->fine = fmodf(d->fine + delta, wrap);
}

dabo_ofdm* dabo_ofdm_create(int mode) {
    int P[6];
    if (dabo_ofdm_params(mode, P) != 0) return NULL;
    dabo_ofdm* d = (dabo_ofdm*)calloc(1, sizeof(*d));
    d->mode = mode; d->L = P[0]; d->Tsym = P[1]; d->Tnull = P[2]; d->CP = P[3]; d->N = P[4]; d->K = P[5];
    d->l1_beta = 0.95f; d->l1_nb_samples = 100; d->l1_decimate = 5;
    d->thresh_null_start = 0.35f; d->thresh_null_end = 0.75f;
    d->fine_beta = 0.9f; d->coarse_enabled = 1; d->max_coarse_norm = 0.5f; d->coarse_slow_beta = 0.1f;
    d->impulse_thresh_db = 20.0f; d->impulse_dist_prob = 0.15f;
    d->state = ST_FINDING_NULL; d->keep = 1;
    const size_t N = (size_t)d->N;
    d->null_ring = (cf*)calloc((size_t)d->Tnull, sizeof(cf));
    d->corr = (cf*)calloc((size_t)(d->Tnull + d->Tsym), sizeof(cf));
    d->frame_cap = (size_t)d->L*(size_t)d->Tsym + (size_t)d->Tnull;
    d->frame = (cf*)calloc(d->frame_cap, sizeof(cf));
    d->prs_fft_conj = (cf*)calloc(N, sizeof(cf)); d->prs_time_ref = (cf*)calloc(N, sizeof(cf));
    d->fftbuf = (cf*)calloc(N, sizeof(cf)); d->ifftbuf = (cf*)calloc(N, sizeof(cf));
    d->spectra = (cf*)calloc(N*(size_t)d->L, sizeof(cf));
    d->impulse = (float*)calloc(N, sizeof(float)); d->freq_resp = (float*)calloc(N, sizeof(float));
    d->phase_err = (float*)calloc((size_t)d->L, sizeof(float));
    d->cmap = (int*)calloc((size_t)d->K, sizeof(int));
    d->plan = fft_make(d->N);
    dabo_carrier_map(d->N, d->K, d->cmap);
    cf* prs = (cf*)calloc(N, sizeof(cf));
    dabo_prs_fft(mode, (float*)prs, d->N);
    /* ofdm_demodulator.cpp:128-140 */
    for (size_t i = 0; i < N; i++) { d->prs_fft_conj[i].re = prs[i].re; d->prs_fft_conj[i].im = -prs[i].im; }
    for (size_t i = 0; i + 1 < N; i++) {           /* CalculateRelativePhase: conj(X[i])*X[i+1] */
        d->prs_time_ref[i].re = prs[i].re*prs[i+1].re + prs[i].im*prs[i+1].im;
        d->prs_time_ref[i].im = prs[i].re*prs[i+1].im - prs[i].im*prs[i+1].re;
    }
    d->prs_time_ref[N-1].re = 0; d->prs_time_ref[N-1].im = 0;
    fft_exec(d->plan, d->prs_time_ref, d->prs_time_ref, 1);
    for (size_t i = 0; i < N; i++) d->prs_time_ref[i].im = -d->prs_time_ref[i].im;
    free(prs);
    return d;
}

void dabo_ofdm_destroy(dabo_ofdm* d) {
    if (!d) return;
    while (d->q_head) { frame_node* n = d->q_head; d->q_head = n->next; free(n); }
    free(d->null_ring); free(d->corr); free(d->frame); free(d->prs_fft_conj); free(d->prs_time_ref);
    free(d->fftbuf); free(d->ifftbuf); free(d->spectra); free(d->impulse); free(d->freq_resp); free(d->phase_err);
    free(d->cmap); fft_free(d->plan); free(d->scratch); free(d);
}
void dabo_ofdm_set_config(dabo_ofdm* d, const dabo_ofdm_config* c) {
    d->l1_beta = c->signal_l1_update_beta; d->l1_nb_samples = c->signal_l1_nb_samples; d->l1_decimate = c->signal_l1_nb_decimate;
    d->thresh_null_start = c->null_thresh_start; d->thresh_null_end = c->null_thresh_end;
    d->fine_beta = c->fine_freq_update_beta; d->coarse_enabled = c->is_coarse_freq_correction;
    d->max_coarse_norm = c->max_coarse_freq_correction_norm; d->coarse_slow_beta = c->coarse_freq_slow_beta;
    d->impulse_thresh_db = c->impulse_peak_threshold_db; d->impulse_dist_prob = c->impulse_peak_distance_probability;
}
int dabo_ofdm_frame_bits(const dabo_ofdm* d) { return (d->L - 1)*d->K*2; }
void dabo_ofdm_keep_frames(dabo_ofdm* d, int keep) { d->keep = keep; }

static void ofdm_reset(dabo_ofdm* d) {         /* ofdm_demodulator.cpp:277-289 */
    d->state = ST_FINDING_NULL; d->corr_len = 0; d->frames_desync++;
    d->coarse_found = 0; d->coarse = 0; d->fine = 0; d->fine_time_offset = 0;
}

/* ofdm_demodulator.cpp:650-766 + 581-639 executed inline (canonical order) */
static void process_frame(dabo_ofdm* d) {
    const size_t N = (size_t)d->N, T = (size_t)d->Tsym, CP = (size_t)d->CP, K = (size_t)d->K;
    const float f = d->coarse + d->fine;
    for (int s = 0; s <= d->L; s++) {
        cf* sym = d->frame + (size_t)s*T;
        const size_t len = (s < d->L) ? T : (size_t)d->Tnull;
        const float dt0 = (float)(s*d->Tsym)*f;
        apply_pll(sym, sym, len, f, dt0);
    }
    float total = 0.0f;
    for (int s = 0; s < d->L; s++) {
        const cf* sym = d->frame + (size_t)s*T;
        const cf e = conj_mul_sum(sym + N, sym, CP);
        total += atan2f(e.im, e.re);
    }
    {   /* coordinator: ofdm_demodulator.cpp:608-618, 779-824 */
        const float avg = total/(float)d->L;
        const float err = (1.0f/(float)d->N)*avg/(2.0f*(float)M_PI);
        update_fine(d, -d->fine_beta*err);
    }
    for (int s = 0; s < d->L; s++) fft_exec(d->plan, d->frame + (size_t)s*T + CP, d->spectra + (size_t)s*N, 0);
    frame_node* node = NULL;
    if (d->keep) {
        node = (frame_node*)malloc(sizeof(frame_node) + (size_t)dabo_ofdm_frame_bits(d));
        node->next = NULL;
    }
    cf* vec = d->fftbuf;   /* reuse as dqpsk scratch (K <= N) */
    for (int l = 0; l + 1 < d->L; l++) {
        const cf* X0 = d->spectra + (size_t)l*N;       /* in1 */
        const cf* X1 = d->spectra + (size_t)(l+1)*N;   /* in0 */
        size_t idx = 0;
        for (int i = -(int)(K/2); i <= (int)(K/2); i++) {
            if (i == 0) continue;
            const size_t b = (size_t)((d->N + i) % d->N);
            vec[idx].re = X0[b].re*X1[b].re + X0[b].im*X1[b].im;
            vec[idx].im = X0[b].im*X1[b].re - X0[b].re*X1[b].im;
            idx++;
        }
        if (node) {
            int8_t* out = node->bits + (size_t)l*2u*K;
            for (size_t i = 0; i < K; i++) {
                const cf v = vec[d->cmap[i]];
                const float A = fmaxf(fabsf(v.re), fabsf(v.im));
                out[i]   = (int8_t)((v.re/A)*-127.0f);
                out[i+K] = (int8_t)((v.im/A)*127.0f);
            }
        }
    }
    d->frames_read++;
    if (node) {
        node->coarse = d->coarse; node->fine = d->fine; node->time_offset = d->fine_time_offset;
        if (d->q_tail) d->q_tail->next = node; else d->q_head = node;
        d->q_tail = node;
    }
}

static size_t find_null(dabo_ofdm* d, const cf* buf, size_t n) {       /* :291-347 */
    const int N = (int)n, K = d->l1_nb_samples, M = N - K;
    const float t0 = d->l1_avg*d->thresh_null_start, t1 = d->l1_avg*d->thresh_null_end;
    int nb_read = N;
    for (int i = 0; i < M; i += K) {
        const float a = l1_average(buf + i, (size_t)K);
        if (d->null_start_found) { if (a > t1) { d->null_end_found = 1; nb_read = i + K; break; } }
        else if (a < t0) d->null_start_found = 1;
    }
    const size_t cap = (size_t)d->Tnull;
    for (int i = 0; i < nb_read; i++) { d->null_ring[d->ring_index++] = buf[i]; d->ring_index %= cap; }
    d->ring_len += (size_t)nb_read; if (d->ring_len > cap) d->ring_len = cap;
    if (!d->null_end_found) return (size_t)nb_read;
    const size_t L = d->ring_len, start = d->ring_index;
    for (size_t i = 0; i < L; i++) d->corr[i] = d->null_ring[(i + start) % cap];
    d->null_start_found = 0; d->null_end_found = 0;
    d->corr_len = L; d->ring_len = 0; d->state = ST_READING_NULL_PRS;
    return (size_t)nb_read;
}

static void coarse_sync(dabo_ofdm* d) {                                  /* :360-471 */
    if (!d->coarse_enabled) { d->coarse = 0; d->state = ST_FINE_TIME; return; }
    const int N = d->N, M = N/2;
    const cf* prs = d->corr + d->Tnull;
    fft_exec(d->plan, prs, d->fftbuf, 0);
    for (int i = 0; i < N-1; i++) {
        const cf a = d->fftbuf[i], b = d->fftbuf[i+1];
        d->fftbuf[i].re = a.re*b.re + a.im*b.im;
        d->fftbuf[i].im = a.re*b.im - a.im*b.re;
    }
    d->fftbuf[N-1].re = 0; d->fftbuf[N-1].im = 0;
    fft_exec(d->plan, d->fftbuf, d->ifftbuf, 1);
    for (int i = 0; i < N; i++) {
        const cf a = d->ifftbuf[i], b = d->prs_time_ref[i];
        d->ifftbuf[i].re = a.re*b.re - a.im*b.im;
        d->ifftbuf[i].im = a.re*b.im + a.im*b.re;
    }
    fft_exec(d->plan, d->ifftbuf, d->fftbuf, 0);
    for (int i = 0; i < N; i++) d->freq_resp[i] = 20.0f*log10f(cabs_f(d->fftbuf[(i + M) % N]));
    int maxoff = (int)(d->max_coarse_norm*(float)N);
    if (maxoff < 0) maxoff = 0;
    if (maxoff > M) maxoff = M;
    int max_index = -maxoff;
    float max_value = d->freq_resp[max_index + M];
    for (int i = -maxoff; i <= maxoff; i++) {
        const int k = i + M;
        if (k == N) continue;
        if (d->freq_resp[k] > max_value) { max_value = d->freq_resp[k]; max_index = i; }
    }
    float mag[3]; int pk[3];
    for (int j = 0; j < 3; j++) {
        int idx = max_index - 1 + j;
        if (idx < -maxoff) idx = -maxoff;
        if (idx > maxoff) idx = maxoff;
        int k = idx + M;
        if (k >= N) k = N-1;
        mag[j] = powf(10.0f, d->freq_resp[k]/20.0f);
        pk[j] = k - M;
    }
    const float sum = mag[0] + mag[1] + mag[2];
    float lerp = 0.0f;
    for (int j = 0; j < 3; j++) lerp += (float)pk[j]*mag[j]/sum;
    const float predicted = -lerp/(float)N;
    const float error = predicted - d->coarse;
    const int large = fabsf(error) > 1.5f/(float)N;
    const float beta = (large || !d->coarse_found) ? 1.0f : d->coarse_slow_beta;
    const float delta = beta*error;
    d->coarse += delta;
    d->coarse_found = 1;
    update_fine(d, -delta);
    d->state = ST_FINE_TIME;
}

static void fine_time_sync(dabo_ofdm* d) {                               /* :473-548 */
    const int N = d->N;
    const cf* prs = d->corr + d->Tnull;
    const float f = d->coarse + d->fine;
    apply_pll(prs, d->ifftbuf, (size_t)N, f, 0.0f);
    fft_exec(d->plan, d->ifftbuf, d->fftbuf, 0);
    for (int i = 0; i < N; i++) {
        const cf a = d->fftbuf[i], b = d->prs_fft_conj[i];
        d->fftbuf[i].re = a.re*b.re - a.im*b.im;
        d->fftbuf[i].im = a.re*b.im + a.im*b.re;
    }
    fft_exec(d->plan, d->fftbuf, d->ifftbuf, 1);
    for (int i = 0; i < N; i++) d->impulse[i] = 20.0f*log10f(cabs_f(d->ifftbuf[i]));
    float avg = 0.0f, maxv = d->impulse[0];
    int maxi = 0;
    for (int i = 0; i < N; i++) {
        const float v = d->impulse[i];
        const int dist = abs(d->CP - i);
        const float nd = (float)dist/(float)d->Tsym;
        const float w = 1.0f - (1.0f - d->impulse_dist_prob)*nd;
        const float wv = w*v;
        avg += v;
        if (wv > maxv) { maxv = wv; maxi = i; }
    }
    avg /= (float)N;
    if ((maxv - avg) < d->impulse_thresh_db) { ofdm_reset(d); return; }
    const int offset = maxi - d->CP;
    const size_t start = (size_t)(d->Tnull + offset), len = (size_t)(d->Tsym - offset);
    memcpy(d->frame, d->corr + start, len*sizeof(cf));
    d->frame_fill = len;
    d->corr_len = 0;
    d->fine_time_offset = offset;
    d->state = ST_READING_SYMBOLS;
}

static void process_block(dabo_ofdm* d, const cf* buf, size_t n) {       /* Process, :235-275 */
    {   /* UpdateSignalAverage :934-950 */
        const size_t Kn = (size_t)d->l1_nb_samples;
        if (n >= Kn) {
            const size_t M = n - Kn, Lstep = Kn*(size_t)d->l1_decimate;
            for (size_t i = 0; i < M; i += Lstep)
                d->l1_avg = d->l1_beta*d->l1_avg + (1.0f - d->l1_beta)*l1_average(buf + i, Kn);
        }
    }
    size_t cur = 0;
    while (cur < n) {
        const cf* b = buf + cur; const size_t rem = n - cur;
        switch (d->state) {
        case ST_FINDING_NULL: cur += find_null(d, b, rem); break;
        case ST_READING_NULL_PRS: {
            const size_t cap = (size_t)(d->Tnull + d->Tsym);
            const size_t need = cap - d->corr_len, take = rem < need ? rem : need;
            memcpy(d->corr + d->corr_len, b, take*sizeof(cf));
            d->corr_len += take; cur += take;
            if (d->corr_len == cap) d->state = ST_COARSE;
        } break;
        case ST_COARSE: coarse_sync(d); break;
        case ST_FINE_TIME: fine_time_sync(d); break;
        case ST_READING_SYMBOLS: {
            const size_t need = d->frame_cap - d->frame_fill, take = rem < need ? rem : need;
            memcpy(d->frame + d->frame_fill, b, take*sizeof(cf));
            d->frame_fill += take; cur += take;
            if (d->frame_fill == d->frame_cap) {
                memcpy(d->corr, d->frame + (size_t)d->L*(size_t)d->Tsym, (size_t)d->Tnull*sizeof(cf));
                d->corr_len = (size_t)d->Tnull;
                d->state = ST_READING_NULL_PRS;
                process_frame(d);
                d->frame_fill = 0;
            }
        } break;
        }
    }
}

void dabo_ofdm_process_c32(dabo_ofdm* d, const float* iq, int n) { process_block(d, (const cf*)iq, (size_t)n); }

void dabo_ofdm_process_u8(dabo_ofdm* d, const uint8_t* iq, int n) {   /* app_iq_readers.h:23-43,72-87 */
    if (d->scratch_cap < (size_t)n) { d->scratch = (cf*)realloc(d->scratch, sizeof(cf)*(size_t)n); d->scratch_cap = (size_t)n; }
    const float scale = 1.0f/127.5f;
    for (int i = 0; i < n; i++) {
        d->scratch[i].re = ((float)iq[2*i] - 127.5f)*scale;
        d->scratch[i].im = ((float)iq[2*i+1] - 127.5f)*scale;
    }
    process_block(d, d->scratch, (size_t)n);
}

int dabo_ofdm_pop_frame(dabo_ofdm* d, int8_t* out, float* cf2, int* toff) {
    frame_node* n = d->q_head;
    if (!n) return 0;
    d->q_head = n->next; if (!d->q_head) d->q_tail = NULL;
    memcpy(out, n->bits, (size_t)dabo_ofdm_frame_bits(d));
    if (cf2) { cf2[0] = n->coarse; cf2[1] = n->fine; }
    if (toff) *toff = n->time_offset;
    free(n);
    return 1;
}

void dabo_ofdm_get_state(const dabo_ofdm* d, int* s4, float* f3) {
    s4[0] = d->state; s4[1] = d->frames_read; s4[2] = d->frames_desync; s4[3] = d->fine_time_offset;
    f3[0] = d->l1_avg; f3[1] = d->coarse; f3[2] = d->fine;
}

double dabo_time_ofdm_u8(int mode, const uint8_t* iq, long n_samples, int block_size, int repeat, int* frames_out) {
    dabo_ofdm* d = dabo_ofdm_create(mode);
    if (!d) return -1.0;
    d->keep = 0;
    struct timespec t0, t1;
    clock_gettime(CLOCK_MONOTONIC, &t0);
    for (int r = 0; r < repeat; r++)
        for (long off = 0; off < n_samples; off += block_size) {
            const long n = (n_samples - off < block_size) ? (n_samples - off) : block_size;
            dabo_ofdm_process_u8(d, iq + 2*off, (int)n);
        }
    clock_gettime(CLOCK_MONOTONIC, &t1);
    if (frames_out) *frames_out = d->frames_read;
    dabo_ofdm_destroy(d);
    return (double)(t1.tv_sec - t0.tv_sec) + 1e-9*(double)(t1.tv_nsec - t0.tv_nsec);
}
