// tables.cuh -- constant tables of the DAB channel code (device constant memory + host builders)
#pragma once
#include "common.cuh"

// ---------------------------------------------------------------------------------------------
// Puncturing.  Reference: dab/constants/puncture_codes.h:42-69 (count-table form of EN 300 401
// table 13).  PI_i keeps 8+i of every 32 mother bits: every 4-bit group keeps 1+(i-1)/8 bits and
// the groups 0,4,2,6,1,5,3,7 (in that order) receive the (i-1)%8+1 extra bits.
// Row 0 is the 24-bit tail code PI_X (2 of every 4).
// Per row: cnt  = eight 4-bit fields (bits kept in group g)
//          pref = eight 8-bit fields (bits kept before group g inside the 32-bit period)
//          K    = bits kept per period of 8 groups
// ---------------------------------------------------------------------------------------------
__constant__ uint32_t c_pi_cnt[25];
__constant__ uint64_t c_pi_pref[25];
__constant__ uint32_t c_pi_K[25];

static void host_pi_counts(int pi, int cnt[8]) {
    if (pi == 0) {
        for (int g = 0; g < 8; g++) cnt[g] = 2;
        return;
    }
    static const int order[8] = {0, 4, 2, 6, 1, 5, 3, 7};
    const int base = 1 + (pi - 1) / 8;
    for (int g = 0; g < 8; g++) cnt[g] = base;
    for (int k = 0; k <= (pi - 1) % 8; k++) cnt[order[k]]++;
}

// Branch table: lane (= half-state s) -> four int8 expected symbols packed in one word.
// Reference: VIT/viterbi_branch_table.h:45-55 with G = {109,79,83,109} (dab_viterbi_decoder.cpp:18-25)
__constant__ uint32_t c_branch[32];

// CRC tables (MSB-first, crc.h:46-67): CCITT 0x1021 (FIB, AU) and the fire code 0x782F
__constant__ uint16_t c_crc_ccitt[256];
__constant__ uint16_t c_crc_fire[256];

// x^(8m) mod the CCITT polynomial, m = 0..34559: the weight of a partial CRC that is followed by m more bytes (k_dabplus splits
// the CRC of an access unit over the 32 lanes of a warp).  An access unit lies inside one superframe of at most 5 * 6912 bytes,
// so m stays below that (static_assert next to crc16_ccitt_warp).  In global memory: every lane reads a different entry.
#define CRC_XP8_ENTRIES 34560
__device__ uint16_t g_crc_xp8[CRC_XP8_ENTRIES];

// Time de-interleaver: age (0 = newest CIF) of the CIF that carries bit i of the oldest complete
// logical frame, i mod 16.  Reference: dab/msc/cif_deinterleaver.cpp:8-11, 62-68 (15 - offset).
__constant__ uint8_t c_ti_age[16];

// GF(2^8)/0x11D exp/log tables.  Reference: reed_solomon_decoder.cpp:108-121
__constant__ uint8_t c_gf_exp[512];
__constant__ uint8_t c_gf_log[256];

// The lookup tables k_dabplus / k_rs_batch / k_packet_fec keep in shared memory, built once on the host and copied by every CTA
// with 16-byte loads (reading the __constant__ tables above with a different index per lane serialises in the constant cache:
// 23 % of k_dabplus's stall samples went there).
struct DpTables {
    uint8_t gf_ex[512];
    uint8_t gf_lg[256];
    uint16_t crc_ccitt[256];
    uint16_t crc_fire[256];
    // branch-free x * alpha^r: gf_exz[gf_lgx[x] + r] with log(0) mapped past the end of the exp table
    uint16_t gf_lgx[256];
    uint8_t gf_exz[528];
    // x -> x * alpha^r for the roots r = 2..9 of the DAB+ code: one lookup per Horner step (root 0 needs none, root 1 is a shift)
    uint8_t gf_mulr[8][256];
};
static_assert(sizeof(DpTables) % 16 == 0, "copied in 16-byte pieces");
__device__ __align__(16) DpTables g_dp_tables;

static int upload_constant_tables() {
    uint32_t cnt[25], K[25];
    uint64_t pref[25];
    for (int pi = 0; pi < 25; pi++) {
        int c[8];
        host_pi_counts(pi, c);
        uint32_t cw = 0;
        uint64_t pw = 0;
        int acc = 0;
        for (int g = 0; g < 8; g++) {
            cw |= uint32_t(c[g]) << (4 * g);
            pw |= uint64_t(acc) << (8 * g);
            acc += c[g];
        }
        cnt[pi] = cw;
        pref[pi] = pw;
        K[pi] = uint32_t(acc);
    }
    CUDA_TRY(cudaMemcpyToSymbol(c_pi_cnt, cnt, sizeof(cnt)));
    CUDA_TRY(cudaMemcpyToSymbol(c_pi_pref, pref, sizeof(pref)));
    CUDA_TRY(cudaMemcpyToSymbol(c_pi_K, K, sizeof(K)));

    static const uint8_t G[4] = {109, 79, 83, 109};
    uint32_t branch[32];
    for (int s = 0; s < 32; s++) {
        uint32_t w = 0;
        for (int r = 0; r < 4; r++) {
            const unsigned v = (unsigned(s) << 1) & G[r];
            const int par = __builtin_parity(v);
            const int8_t b = par ? 127 : -127;
            w |= uint32_t(uint8_t(b)) << (8 * r);
        }
        branch[s] = w;
    }
    CUDA_TRY(cudaMemcpyToSymbol(c_branch, branch, sizeof(branch)));

    uint16_t t1[256], t2[256];
    for (int i = 0; i < 256; i++) {
        uint16_t a = uint16_t(i << 8), b = uint16_t(i << 8);
        for (int j = 0; j < 8; j++) {
            a = (a & 0x8000) ? uint16_t((a << 1) ^ 0x1021) : uint16_t(a << 1);
            b = (b & 0x8000) ? uint16_t((b << 1) ^ 0x782F) : uint16_t(b << 1);
        }
        t1[i] = a;
        t2[i] = b;
    }
    CUDA_TRY(cudaMemcpyToSymbol(c_crc_ccitt, t1, sizeof(t1)));
    CUDA_TRY(cudaMemcpyToSymbol(c_crc_fire, t2, sizeof(t2)));
    {
        static uint16_t xp[CRC_XP8_ENTRIES];
        uint16_t v = 1;     // the polynomial "1"; appending a zero byte multiplies by x^8: one table step
        for (int m = 0; m < CRC_XP8_ENTRIES; m++) {
            xp[m] = v;
            v = uint16_t((v << 8) ^ t1[v >> 8]);
        }
        CUDA_TRY(cudaMemcpyToSymbol(g_crc_xp8, xp, sizeof(xp)));
    }

    static const uint8_t TI[16] = {0, 8, 4, 12, 2, 10, 6, 14, 1, 9, 5, 13, 3, 11, 7, 15};
    uint8_t age[16];
    for (int i = 0; i < 16; i++) age[i] = uint8_t(15 - TI[i]);
    CUDA_TRY(cudaMemcpyToSymbol(c_ti_age, age, sizeof(age)));

    uint8_t ex[512], lg[256];
    int sr = 1;
    lg[0] = 255;
    for (int i = 0; i < 255; i++) {
        lg[sr] = uint8_t(i);
        ex[i] = uint8_t(sr);
        sr <<= 1;
        if (sr & 0x100) sr ^= 0x11D;
        sr &= 255;
    }
    for (int i = 255; i < 512; i++) ex[i] = ex[i - 255];
    ex[255] = ex[0];
    CUDA_TRY(cudaMemcpyToSymbol(c_gf_exp, ex, sizeof(ex)));
    CUDA_TRY(cudaMemcpyToSymbol(c_gf_log, lg, sizeof(lg)));
    {
        static DpTables T;
        memcpy(T.gf_ex, ex, sizeof(ex));
        memcpy(T.gf_lg, lg, sizeof(lg));
        memcpy(T.crc_ccitt, t1, sizeof(t1));
        memcpy(T.crc_fire, t2, sizeof(t2));
        for (int i = 0; i < 256; i++) T.gf_lgx[i] = i ? uint16_t(lg[i]) : uint16_t(512);
        for (int i = 0; i < 528; i++) T.gf_exz[i] = (i < 510) ? ex[i] : uint8_t(0);
        for (int r = 2; r < 10; r++)
            for (int x = 0; x < 256; x++) T.gf_mulr[r - 2][x] = x ? ex[lg[x] + r] : uint8_t(0);
        CUDA_TRY(cudaMemcpyToSymbol(g_dp_tables, &T, sizeof(T)));
    }
    return DABGPU_OK;
}

// Energy dispersal PRBS x^9 + x^5 + 1, all-ones start, MSB-first bytes packed big-endian into words
// (word w = bytes 4w..4w+3, byte 4w in bits 31..24).  Reference: additive_scrambler.h:10-36
static void host_prbs_words(std::vector<uint32_t>& out, size_t n_words) {
    out.resize(n_words);
    uint16_t reg = 0xFFFF;
    for (size_t w = 0; w < n_words; w++) {
        uint32_t v = 0;
        for (int i = 0; i < 32; i++) {
            const uint32_t b = ((reg >> 8) ^ (reg >> 4)) & 1u;
            v = (v << 1) | b;
            reg = uint16_t((reg << 1) | b);
        }
        out[w] = v;
    }
}

// ---------------------------------------------------------------------------------------------
// Protection profiles -> (PI, mother bits) schedule.
// Reference: dab/constants/subchannel_protection_tables.h:21-154, dab/msc/msc_decoder.cpp:77-154
// (EN 300 401 tables 8/15 for UEP, tables 9/10/18/20 for EEP).
// ---------------------------------------------------------------------------------------------
struct Schedule {
    int n_seg = 0;
    int pi[DABGPU_MAX_SEGMENTS] = {0, 0, 0, 0, 0};
    int bits[DABGPU_MAX_SEGMENTS] = {0, 0, 0, 0, 0};
    int total_steps() const {
        int s = 0;
        for (int i = 0; i < n_seg; i++) s += bits[i] / 4;
        return s;
    }
    int punctured_bits() const {
        int total = 0;
        for (int i = 0; i < n_seg; i++) {
            int c[8];
            host_pi_counts(pi[i], c);
            const int groups = bits[i] / 4;
            for (int g = 0; g < groups; g++) total += c[g % 8];
        }
        return total;
    }
};

// UEP table rows as L1..L4 / PI1..PI4 (row order of EN 300 401 table 8: bit rate ascending, protection level 5..1)
static const uint8_t kUepBlocks[64][4] = {
    {3, 4, 17, 0},    {3, 3, 18, 0},    {3, 4, 14, 3},    {3, 4, 14, 3},    {3, 5, 13, 3},    {4, 3, 26, 3},    {3, 4, 26, 3},    {3, 4, 26, 3},
    {3, 4, 26, 3},    {3, 5, 25, 3},    {6, 10, 23, 3},   {6, 10, 23, 3},   {6, 12, 21, 3},   {6, 10, 23, 3},   {6, 9, 31, 2},    {6, 9, 33, 0},
    {6, 12, 27, 3},   {6, 10, 29, 3},   {6, 11, 28, 3},   {6, 10, 41, 3},   {6, 10, 41, 3},   {6, 11, 40, 3},   {6, 10, 41, 3},   {6, 10, 41, 3},
    {7, 9, 53, 3},    {7, 10, 52, 3},   {6, 12, 51, 3},   {6, 10, 53, 3},   {6, 13, 50, 3},   {14, 17, 50, 3},  {11, 21, 49, 3},  {11, 23, 47, 3},
    {11, 21, 49, 3},  {12, 19, 62, 3},  {11, 21, 61, 3},  {11, 22, 60, 3},  {11, 21, 61, 3},  {11, 20, 62, 3},  {11, 19, 87, 3},  {11, 23, 83, 3},
    {11, 24, 82, 3},  {11, 21, 85, 3},  {11, 22, 84, 3},  {11, 20, 110, 3}, {11, 22, 108, 3}, {11, 24, 106, 3}, {11, 20, 110, 3}, {11, 21, 109, 3},
    {12, 22, 131, 3}, {12, 26, 127, 3}, {11, 20, 134, 3}, {11, 22, 132, 3}, {11, 24, 130, 3}, {11, 24, 154, 3}, {11, 24, 154, 3}, {11, 27, 151, 3},
    {11, 22, 156, 3}, {11, 26, 152, 3}, {11, 26, 200, 3}, {11, 25, 201, 3}, {11, 26, 200, 3}, {11, 27, 247, 3}, {11, 24, 250, 3}, {12, 28, 245, 3},
};
static const uint8_t kUepCodes[64][4] = {
    {5, 3, 2, 0},     {11, 6, 5, 0},    {15, 9, 6, 8},    {22, 13, 8, 13},  {24, 17, 12, 17}, {5, 4, 2, 3},     {9, 6, 4, 6},     {15, 10, 6, 9},
    {24, 14, 8, 15},  {24, 18, 13, 18}, {5, 4, 2, 3},     {9, 6, 4, 5},     {16, 7, 6, 9},    {23, 13, 8, 13},  {5, 3, 2, 3},     {11, 6, 5, 0},
    {16, 8, 6, 9},    {23, 13, 8, 13},  {24, 18, 12, 18}, {6, 3, 2, 3},     {11, 6, 5, 6},    {16, 8, 6, 7},    {23, 13, 8, 13},  {24, 17, 12, 18},
    {5, 4, 2, 4},     {9, 6, 4, 6},     {16, 9, 6, 10},   {22, 12, 9, 12},  {24, 18, 13, 19}, {5, 4, 2, 5},     {9, 6, 4, 8},     {16, 8, 6, 9},
    {23, 12, 9, 14},  {5, 3, 2, 4},     {11, 6, 5, 7},    {16, 9, 6, 10},   {22, 12, 9, 14},  {24, 17, 13, 19}, {5, 4, 2, 4},     {11, 6, 5, 9},
    {16, 8, 6, 11},   {22, 11, 9, 13},  {24, 18, 12, 19}, {6, 4, 2, 5},     {10, 6, 4, 9},    {16, 10, 6, 11},  {22, 13, 9, 13},  {24, 20, 13, 24},
    {8, 6, 2, 6},     {12, 8, 4, 11},   {16, 10, 7, 9},   {24, 16, 10, 15}, {24, 20, 12, 20}, {6, 5, 2, 5},     {12, 9, 5, 10},   {16, 10, 7, 10},
    {24, 14, 10, 13}, {24, 19, 14, 18}, {8, 5, 2, 6},     {13, 9, 5, 10},   {24, 17, 9, 17},  {8, 6, 2, 7},     {16, 9, 7, 10},   {24, 20, 14, 23},
};

static int make_schedule(const dabgpu_subchannel& sc, Schedule* out) {
    Schedule s;
    if (sc.is_uep) {
        if (sc.uep_prot_index < 0 || sc.uep_prot_index >= 64) return set_error(DABGPU_ERR_INVALID, "UEP index %d out of range", sc.uep_prot_index);
        for (int i = 0; i < 4; i++) {
            const int L = kUepBlocks[sc.uep_prot_index][i];
            if (L == 0) continue;  // update() with zero requested symbols does nothing (dab_viterbi_decoder.cpp:152)
            s.pi[s.n_seg] = kUepCodes[sc.uep_prot_index][i];
            s.bits[s.n_seg] = 128 * L;
            s.n_seg++;
        }
    } else {
        if (sc.eep_prot_level < 0 || sc.eep_prot_level > 3) return set_error(DABGPU_ERR_INVALID, "EEP level %d out of range", sc.eep_prot_level);
        int L1, L2, p1, p2;
        const int lv = sc.eep_prot_level;
        if (!sc.eep_type_b) {
            static const int mult[4] = {12, 8, 6, 4};
            static const int m1[4] = {6, 2, 6, 4}, m2[4] = {0, 4, 0, 2};
            static const int pa[4] = {24, 14, 8, 3}, pb[4] = {23, 13, 7, 2};
            if (sc.length == 8) {  // GetEEPDescriptor keys the 2-A n=1 row on the length alone (subchannel_protection_tables.h:145-154)
                L1 = 5; L2 = 1; p1 = 13; p2 = 12;
            } else {
                const int n = sc.length / mult[lv];
                L1 = m1[lv] * n - 3; L2 = m2[lv] * n + 3; p1 = pa[lv]; p2 = pb[lv];
            }
        } else {
            static const int mult[4] = {27, 21, 18, 15};
            static const int pa[4] = {10, 6, 4, 2}, pb[4] = {9, 5, 3, 1};
            const int n = sc.length / mult[lv];
            L1 = 24 * n - 3; L2 = 3; p1 = pa[lv]; p2 = pb[lv];
        }
        if (L1 < 0 || L2 < 0) return set_error(DABGPU_ERR_INVALID, "sub-channel length %d too small for the EEP profile", sc.length);
        s.pi[0] = p1; s.bits[0] = 128 * L1;
        s.pi[1] = p2; s.bits[1] = 128 * L2;
        s.n_seg = 2;
    }
    s.pi[s.n_seg] = 0;
    s.bits[s.n_seg] = 24;
    s.n_seg++;
    // A segment whose punctured symbols do not fit what is left of the sub-channel decodes NOTHING and consumes nothing in the
    // reference: depuncture_symbols returns an all-zero result as soon as a 4-bit block runs out of input
    // (dab_viterbi_decoder.cpp:157-161) and DecodeUEP / DecodeEEP carry on with the next update() from the same position
    // (msc_decoder.cpp:86-96, 128-139).  UEP_PROTECTION_TABLE row 34 is listed with 64 CU but needs 84 (rows 33 and 34 are
    // swapped against EN 300 401 table 8): its third segment is skipped and 140 bytes per CIF come out.  Same rule here.
    {
        Schedule f;
        int remaining = sc.length * 64;
        for (int i = 0; i < s.n_seg; i++) {
            int c[8], need = 0;
            host_pi_counts(s.pi[i], c);
            for (int g = 0; g < s.bits[i] / 4; g++) need += c[g % 8];
            if (need > remaining) continue;
            remaining -= need;
            f.pi[f.n_seg] = s.pi[i];
            f.bits[f.n_seg] = s.bits[i];
            f.n_seg++;
        }
        s = f;
    }
    if (s.total_steps() < 6 + 8) return set_error(DABGPU_ERR_INVALID, "sub-channel of %d CU is too small for its protection profile", sc.length);
    *out = s;
    return DABGPU_OK;
}
