// dabplus.cuh -- DAB+ audio superframe stage and Reed-Solomon decoder.
//   AAC_Frame_Processor::{Process,CalculateFirecode,AccumulateFrame,ProcessSuperFrame,ReedSolomonDecode}
//       dab/audio/aac_frame_processor.cpp:126-362
//   Reed_Solomon_Decoder::Decode -> decode_rs_char   dab/algorithms/reed_solomon_decoder.cpp:192-477
//       GF(2^8) poly 0x11D, fcr 0, prim 1; DAB+ uses 10 roots, pad 135 (aac_frame_processor.cpp:105-111)
//
// One warp per (stream, sub-channel): the per-sub-channel state machine is sequential over the CIFs of
// a frame, the RS codewords of a superframe are decoded one per lane (codeword i = bytes {i + j*N}, so
// lanes read consecutive bytes), corrections are applied in codeword order so the reference's
// "stop at the first uncorrectable codeword" behaviour is preserved.
#pragma once
#include "chan.cuh"

#define RS_MAX_ROOTS 32
#define DP_MAX_EVENTS 16

struct DabPlusSubState { int32_t collect, curr_frame, prev_nb, synced, desync, pad0, pad1, pad2; };
struct DabPlusEvent { int32_t type, a, b, c, d, payload_off, payload_len, pad; };

struct DabPlusDev {
    DabPlusSubState* st;     // [stream][max_subs]
    uint8_t* sf;             // [stream][5*CIF_OUT_STRIDE], sub-channel at 5*out_offset: accumulator of the 5 logical frames
    uint8_t* sf_out;         // same layout: last completed (RS corrected, fire code valid) superframe, what the observers see
    DabPlusEvent* events;    // [stream][max_subs][DP_MAX_EVENTS]
    int32_t* n_events;       // [stream][max_subs]
};

struct DabPlusState {
    DevBuf d_st, d_sf, d_sf_out, d_events, d_nevents, d_rs_cw, d_rs_cnt, d_rs_pos;
    DabPlusDev dev;
    int max_streams = 0, max_subs = 0, nb_cifs = 0;
};

struct GfTables { const uint8_t* ex; const uint8_t* lg; };

__device__ __forceinline__ int gf_mod255(int x) {
    while (x >= 255) { x -= 255; x = (x >> 8) + (x & 255); }
    return x;
}
__device__ __forceinline__ uint8_t gf_mul_dev(const GfTables& T, uint8_t a, uint8_t b) {
    return (a && b) ? T.ex[T.lg[a] + T.lg[b]] : uint8_t(0);
}

// Syndromes S_i = data(alpha^i), Horner from data[0] (reed_solomon_decoder.cpp:232-245).  Returns OR of all S_i.
__device__ int rs_syndromes(const GfTables& T, const uint8_t* data, int stride, int n, int nroots, uint8_t* S) {
    for (int i = 0; i < nroots; i++) S[i] = data[0];
    for (int j = 1; j < n; j++) {
        const uint8_t d = data[size_t(j) * stride];
        for (int i = 0; i < nroots; i++) S[i] = uint8_t(d ^ (S[i] ? T.ex[gf_mod255(T.lg[S[i]] + i)] : 0));
    }
    int any = 0;
    for (int i = 0; i < nroots; i++) any |= S[i];
    return any;
}

// Berlekamp-Massey + Chien + Forney for fcr = 0, prim = 1 (reed_solomon_decoder.cpp:263-466).
// Outputs error locations (incl. pad) and the value to XOR at each location; apply[j] = 0 where the
// reference leaves the data untouched (zero error value or location inside the padding).
__device__ int rs_solve(const GfTables& T, const uint8_t* S, int nroots, int pad, uint8_t* loc, uint8_t* xorval, uint8_t* apply) {
    uint8_t lambda[RS_MAX_ROOTS + 1], b[RS_MAX_ROOTS + 1], t[RS_MAX_ROOTS + 1], omega[RS_MAX_ROOTS + 1], root[RS_MAX_ROOTS];
    for (int i = 0; i <= nroots; i++) { lambda[i] = 0; b[i] = 0; }
    lambda[0] = 1; b[0] = 1;
    int el = 0;
    for (int r = 1; r <= nroots; r++) {
        uint8_t discr = 0;
        for (int i = 0; i < r; i++) discr ^= gf_mul_dev(T, lambda[i], S[r - i - 1]);
        if (discr == 0) {
            for (int i = nroots; i > 0; i--) b[i] = b[i - 1];
            b[0] = 0;
        } else {
            t[0] = lambda[0];
            for (int i = 0; i < nroots; i++) t[i + 1] = uint8_t(lambda[i + 1] ^ gf_mul_dev(T, discr, b[i]));
            if (2 * el <= r - 1) {
                el = r - el;
                const int ld = T.lg[discr];
                for (int i = 0; i <= nroots; i++) b[i] = lambda[i] ? T.ex[gf_mod255(T.lg[lambda[i]] - ld + 255)] : uint8_t(0);
            } else {
                for (int i = nroots; i > 0; i--) b[i] = b[i - 1];
                b[0] = 0;
            }
            for (int i = 0; i <= nroots; i++) lambda[i] = t[i];
        }
    }
    int deg_lambda = 0;
    for (int i = 0; i <= nroots; i++) if (lambda[i]) deg_lambda = i;
    int count = 0;
    for (int i = 1; i <= 255; i++) {
        uint8_t q = 1;
        for (int j = deg_lambda; j > 0; j--) if (lambda[j]) q ^= T.ex[gf_mod255(T.lg[lambda[j]] + (i * j) % 255)];
        if (q != 0) continue;
        root[count] = uint8_t(i);
        loc[count] = uint8_t(i - 1);
        if (++count == deg_lambda) break;
    }
    if (deg_lambda != count) return -1;
    const int deg_omega = deg_lambda - 1;
    for (int i = 0; i <= deg_omega; i++) {
        uint8_t tmp = 0;
        for (int j = i; j >= 0; j--) tmp ^= gf_mul_dev(T, S[i - j], lambda[j]);
        omega[i] = tmp;
    }
    for (int j = count - 1; j >= 0; j--) {
        uint8_t num1 = 0, den = 0;
        for (int i = deg_omega; i >= 0; i--) if (omega[i]) num1 ^= T.ex[gf_mod255(T.lg[omega[i]] + (i * root[j]) % 255)];
        const uint8_t num2 = T.ex[gf_mod255(255 - root[j])];
        const int top = min(deg_lambda, nroots - 1) & ~1;
        for (int i = top; i >= 0; i -= 2) if (lambda[i + 1]) den ^= T.ex[gf_mod255(T.lg[lambda[i + 1]] + (i * root[j]) % 255)];
        apply[j] = (num1 != 0 && loc[j] >= pad) ? 1 : 0;
        // index arithmetic kept as in the reference (log(0) = 255) so that even den == 0 gives the same byte
        xorval[j] = T.ex[gf_mod255(int(T.lg[num1]) + int(T.lg[num2]) + 255 - int(T.lg[den]))];
    }
    return count;
}

#define DP_WARPS 4
#define DP_SF_SMEM 1920   // superframes up to 128 kbit/s (5 x 384 bytes) are staged in shared memory per warp
struct DpShared : DpTables {
    __align__(16) uint8_t sfbuf[DP_WARPS][DP_SF_SMEM];
};

__device__ __forceinline__ void dp_load_shared(DpShared& sh) {
    const uint4* src = reinterpret_cast<const uint4*>(&g_dp_tables);
    uint4* dst = reinterpret_cast<uint4*>(static_cast<DpTables*>(&sh));
    for (int i = threadIdx.x; i < int(sizeof(DpTables) / 16); i += blockDim.x) dst[i] = src[i];
    __syncthreads();
}

__device__ __forceinline__ uint16_t crc16_tab(const uint16_t* tab, const uint8_t* p, int n, uint16_t init, uint16_t xorout) {
    uint32_t crc = init;
    for (int i = 0; i < n; i++) crc = ((crc << 8) ^ tab[((crc >> 8) ^ p[i]) & 0xFFu]) & 0xFFFFu;
    return uint16_t(crc ^ xorout);
}

// a * b in GF(2)[x] modulo the CCITT polynomial x^16 + x^12 + x^5 + 1
__device__ __forceinline__ uint32_t crc_mulmod(const uint32_t a, const uint32_t b) {
    uint32_t r = 0;
#pragma unroll
    for (int i = 15; i >= 0; i--) {
        r <<= 1;
        if (r & 0x10000u) r ^= 0x11021u;
        if ((b >> i) & 1u) r ^= a;
    }
    return r;
}

// CRC16-CCITT (init 0xFFFF, final inversion; crc.h:46-67) of n bytes by a whole warp: lane l runs the table loop over its chunk
// of ceil(n / 32) bytes (lane 0 carries the initial value), weighs the result with x^(8 * bytes that follow) and the lanes XOR
// their shares.  A 300-byte access unit is a dependent chain of 10 table steps instead of 300.  Every lane returns the CRC.
// Lane 0 reads weight n - ceil(n / 32); n is at most a superframe (5 logical frames of up to CIF_OUT_STRIDE bytes).
static_assert(CRC_XP8_ENTRIES >= 5 * CIF_OUT_STRIDE, "g_crc_xp8 must hold a weight for every access-unit length");
__device__ __forceinline__ uint16_t crc16_ccitt_warp(const uint16_t* tab, const uint8_t* p, const int n, const uint32_t lane) {
    const int c = (n + 31) >> 5;
    const int b0 = min(n, int(lane) * c), b1 = min(n, b0 + c);
    uint32_t crc = (lane == 0u) ? 0xFFFFu : 0u;
    for (int k = b0; k < b1; k++) crc = ((crc << 8) ^ tab[((crc >> 8) ^ p[k]) & 0xFFu]) & 0xFFFFu;
    uint32_t share = (b1 > b0 || lane == 0u) ? crc_mulmod(crc, g_crc_xp8[n - b1]) : 0u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) share ^= __shfl_xor_sync(FULL_MASK, share, o);
    return uint16_t(share ^ 0xFFFFu);
}

__device__ __forceinline__ void dp_emit(DabPlusEvent* ev, int32_t* n_ev, int type, int a, int b, int c, int d, int off, int len) {
    const int k = *n_ev;
    if (k < DP_MAX_EVENTS) {
        ev[k].type = type; ev[k].a = a; ev[k].b = b; ev[k].c = c; ev[k].d = d;
        ev[k].payload_off = off; ev[k].payload_len = len; ev[k].pad = 0;
    }
    *n_ev = k + 1;
}

// read_au_start (aac_frame_processor.cpp:30-72): n 12-bit values MSB first; returns bytes consumed
__device__ int dp_read_au_start(const uint8_t* buf, uint16_t* data, int n) {
    int bitpos = 0;
    for (int i = 0; i < n; i++) {
        unsigned v = 0;
        for (int k = 0; k < 12; k++, bitpos++) v = (v << 1) | ((buf[bitpos >> 3] >> (7 - (bitpos & 7))) & 1u);
        data[i] = uint16_t(v);
    }
    return (bitpos + 7) >> 3;
}

// n bytes by a warp: 8-byte words when the layout allows it (logical frames are multiples of 24 bytes at multiples of 8), all
// loads of a lane issued before its stores
__device__ __forceinline__ void dp_copy_bytes(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, const int n, const uint32_t lane) {
    if (((reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src) | uintptr_t(n)) & 7u) == 0u) {
        const uint2* s8 = reinterpret_cast<const uint2*>(src);
        uint2* d8 = reinterpret_cast<uint2*>(dst);
        const int n8 = n >> 3;
        for (int i0 = 0; i0 < n8; i0 += 128) {
            uint2 v[4];
#pragma unroll
            for (int k = 0; k < 4; k++) { const int i = i0 + int(lane) + 32 * k; if (i < n8) v[k] = s8[i]; }
#pragma unroll
            for (int k = 0; k < 4; k++) { const int i = i0 + int(lane) + 32 * k; if (i < n8) d8[i] = v[k]; }
        }
    } else {
        for (int i = int(lane); i < n; i += 32) dst[i] = src[i];
    }
}

// ProcessSuperFrame for one sub-channel, executed by a full warp.  Returns nothing; state/event side effects.
__device__ void dp_superframe(DpShared& sh, uint8_t* sf_global, uint8_t* sf_out, const int sf_base, const int nb, DabPlusSubState& st,
                              DabPlusEvent* ev, int32_t* n_ev, unsigned long long* counters, const uint32_t lane) {
    const GfTables T{sh.gf_ex, sh.gf_lg};
    const int total = nb * 5;
    const int N = total / 120;
    // stage the superframe in shared memory: syndromes and CRCs walk it byte by byte (a dependent global load per byte otherwise)
    uint8_t* sf = sf_global;
    if (total <= DP_SF_SMEM && (total & 3) == 0 && (reinterpret_cast<uintptr_t>(sf_global) & 3u) == 0) {
        sf = sh.sfbuf[(threadIdx.x >> 5) % DP_WARPS];
        const uint32_t* src = reinterpret_cast<const uint32_t*>(sf_global);
        uint32_t* dst = reinterpret_cast<uint32_t*>(sf);
        for (int i = int(lane); i < total / 4; i += 32) dst[i] = src[i];
        __syncwarp();
    }
    // ReedSolomonDecode (aac_frame_processor.cpp:322-362): codeword i = bytes {i + j*N}.  Eight codewords per pass, four lanes per
    // codeword: lane part q runs the Horner recurrences of ALL ten roots (reed_solomon_decoder.cpp:223-240) over bytes 30q .. 30q+29
    // -- ten independent chains of 30 steps, one table lookup per step (x -> x * alpha^r) -- then moves its partial syndromes to
    // the end of the codeword (times alpha^(30 r (3 - q))) and the four lanes XOR their shares.  The first version ran three
    // chains of 120 steps with two dependent lookups each per lane: the kernel was bound by that latency.
    for (int base = 0; base < N; base += 8) {
        const int i = base + int(lane >> 2);
        const int part = int(lane & 3u);
        uint32_t P[10];
#pragma unroll
        for (int r = 0; r < 10; r++) P[r] = 0u;
        if (i < N) {
            const uint8_t* p = sf + i + 30 * part * N;
#pragma unroll 2
            for (int j = 0; j < 30; j++) {
                const uint32_t d = p[j * N];
                P[0] ^= d;
                P[1] = (((P[1] << 1) ^ ((P[1] & 0x80u) ? 0x11Du : 0u)) ^ d) & 0xFFu;
#pragma unroll
                for (int r = 2; r < 10; r++) P[r] = uint32_t(sh.gf_mulr[r - 2][P[r]]) ^ d;
            }
            if (part < 3) {
#pragma unroll
                for (int r = 1; r < 10; r++) {
                    const int e = (30 * r * (3 - part)) % 255;
                    P[r] = P[r] ? uint32_t(sh.gf_ex[int(sh.gf_lg[P[r]]) + e]) : 0u;
                }
            }
        }
        uint32_t pk0 = P[0] | (P[1] << 8) | (P[2] << 16) | (P[3] << 24), pk1 = P[4] | (P[5] << 8) | (P[6] << 16) | (P[7] << 24), pk2 = P[8] | (P[9] << 8);
#pragma unroll
        for (int o = 1; o <= 2; o <<= 1) {
            pk0 ^= __shfl_xor_sync(FULL_MASK, pk0, o);
            pk1 ^= __shfl_xor_sync(FULL_MASK, pk1, o);
            pk2 ^= __shfl_xor_sync(FULL_MASK, pk2, o);
        }
        uint8_t S[10];
#pragma unroll
        for (int r = 0; r < 10; r++) S[r] = uint8_t((r < 4 ? pk0 : r < 8 ? pk1 : pk2) >> (8 * (r & 3)));
        int cnt = 0;
        uint8_t loc[10], xv[10], ap[10];
        const bool leader = (part == 0) && (i < N);
        if (leader) {
            int any = 0;
#pragma unroll
            for (int r = 0; r < 10; r++) any |= S[r];
            if (any) cnt = rs_solve(T, S, 10, 135, loc, xv, ap);
        }
        const uint32_t fail_mask = __ballot_sync(FULL_MASK, leader && cnt < 0);
        const int first_fail = fail_mask ? ((__ffs(int(fail_mask)) - 1) >> 2) : 8;   // codeword slot inside this pass
        if (leader && int(lane >> 2) < first_fail) {
            for (int j = 0; j < cnt; j++) {
                const int k = int(loc[j]) - 135;
                if (k >= 0 && ap[j]) sf[i + k * N] ^= xv[j];
            }
        }
        __syncwarp();
        if (fail_mask) {
            if (lane == 0) {
                dp_emit(ev, n_ev, DABGPU_EV_RS_ERROR, base + first_fail, N, 0, 0, 0, 0);
                st.desync++;
                atomicAdd(&counters[CNT_SF_RS_FAIL], 1ull);
            }
            return;
        }
    }
    __syncwarp();
    // fire code on the corrected superframe (aac_frame_processor.cpp:179-191, 210-213)
    int ok = 0;
    if (lane == 0) {
        const uint16_t rx = uint16_t((uint16_t(sf[0]) << 8) | sf[1]);
        const uint16_t pred = crc16_tab(sh.crc_fire, sf + 2, 9, 0, 0);
        ok = (rx == pred);
        if (!ok) {
            dp_emit(ev, n_ev, DABGPU_EV_FIRECODE_ERROR, st.curr_frame, rx, pred, 0, 0, 0);
            st.desync++;
            atomicAdd(&counters[CNT_SF_FIRE_FAIL], 1ull);
        }
    }
    ok = __shfl_sync(FULL_MASK, ok, 0);
    if (!ok) return;
    // the accumulator is reused by the following CIFs of this frame: keep the validated superframe for the host
    dp_copy_bytes(sf_out, sf, total, lane);
    // header (aac_frame_processor.cpp:215-279)
    const uint8_t dsc = sf[2];
    const int dac_rate = (dsc >> 6) & 1, sbr = (dsc >> 5) & 1, ch = (dsc >> 4) & 1, ps = (dsc >> 3) & 1, mpeg = dsc & 7;
    int num_aus = 0;
    if (!dac_rate && sbr) num_aus = 2;
    if (dac_rate && sbr) num_aus = 3;
    if (!dac_rate && !sbr) num_aus = 4;
    if (dac_rate && !sbr) num_aus = 6;
    uint16_t au_start[7] = {0, 0, 0, 0, 0, 0, 0};
    const int nb_tbl = dp_read_au_start(sf + 3, &au_start[1], num_aus - 1);
    au_start[num_aus] = uint16_t(110 * N);
    au_start[0] = uint16_t(3 + nb_tbl);
    // access units in order (aac_frame_processor.cpp:281-320): bounds, CRC by the whole warp, events from lane 0
    if (lane == 0) {
        st.desync = 0; st.synced = 1;
        const int surround = (mpeg == 0) ? 0 : (mpeg == 1) ? 1 : (mpeg == 2) ? 2 : (mpeg == 7) ? 3 : 4;
        dp_emit(ev, n_ev, DABGPU_EV_SUPERFRAME_HEADER, dac_rate ? 48000 : 32000, (ps ? 1 : 0) | (sbr ? 2 : 0) | (ch ? 4 : 0), surround, 0, 0, 0);
        atomicAdd(&counters[CNT_SF_OK], 1ull);
    }
    for (int i = 0; i < num_aus; i++) {
        const int nb_data = int(au_start[i + 1]) - int(au_start[i]) - 2;
        if (nb_data < 0 || int(au_start[i + 1]) >= total) break;   // "access unit out of bounds" => return (aac_frame_processor.cpp:289-296)
        const uint8_t* au = sf + au_start[i];
        const uint16_t rx = uint16_t((uint16_t(au[nb_data]) << 8) | au[nb_data + 1]);
        const uint16_t pred = crc16_ccitt_warp(sh.crc_ccitt, au, nb_data, lane);
        if (lane == 0) {
            if (rx != pred) {
                dp_emit(ev, n_ev, DABGPU_EV_AU_CRC_ERROR, i, num_aus, int(rx), int(pred), 0, 0);
                atomicAdd(&counters[CNT_AU_CRC_FAIL], 1ull);
            } else {
                dp_emit(ev, n_ev, DABGPU_EV_ACCESS_UNIT, i, num_aus, 0, 0, sf_base + int(au_start[i]), nb_data);
                atomicAdd(&counters[CNT_AU_OK], 1ull);
            }
        }
    }
}

// AAC_Frame_Processor::Process for one logical frame of n bytes (aac_frame_processor.cpp:126-177), executed by a full
// warp; all lanes keep identical copies of st.
__device__ void dp_process_frame(DpShared& sh, const uint8_t* __restrict__ buf, const int n, DabPlusSubState& st, uint8_t* sf, uint8_t* sf_out,
                                 const int sf_base, DabPlusEvent* ev, int32_t* n_ev, unsigned long long* counters, const uint32_t lane) {
    if (n < 11) return;
    if (st.prev_nb != n) { st.prev_nb = n; st.curr_frame = 0; st.collect = 0; }
    if (st.desync >= 10) { st.desync = 0; st.synced = 0; }
    if (st.synced) st.collect = 1;
    if (!st.collect) {
        int ok = 0;
        if (lane == 0) {
            const uint16_t rx = uint16_t((uint16_t(buf[0]) << 8) | buf[1]);
            const uint16_t pred = crc16_tab(sh.crc_fire, buf + 2, 9, 0, 0);
            ok = (rx == pred);
            if (!ok) dp_emit(ev, n_ev, DABGPU_EV_FIRECODE_ERROR, st.curr_frame, rx, pred, 0, 0, 0);
        }
        ok = __shfl_sync(FULL_MASK, ok, 0);
        if (!ok) return;
        st.collect = 1;
    }
    dp_copy_bytes(sf + size_t(st.curr_frame) * n, buf, n, lane);
    __syncwarp();
    st.curr_frame++;
    if (st.curr_frame == 5) {
        // lane 0 owns the mutable copy during the superframe step, then broadcasts
        dp_superframe(sh, sf, sf_out, sf_base, n, st, ev, n_ev, counters, lane);
        st.desync = __shfl_sync(FULL_MASK, st.desync, 0);
        st.synced = __shfl_sync(FULL_MASK, st.synced, 0);
        st.collect = 0;
        st.curr_frame = 0;
    }
}

// One (stream, sub-channel) work item, executed by a full warp.
__device__ void dp_work_item(DpShared& sh, const ChanDev& C, const DabPlusDev& D, const uint32_t s, const uint32_t sub, const uint32_t lane) {
    const size_t idx = size_t(s) * C.max_subs + sub;
    if (lane == 0) D.n_events[idx] = 0;
    if (!C.status[2 * s] || sub >= C.n_subs[s]) return;
    const SubCfgDev cfg = C.subcfg[idx];
    if (!cfg.is_dabplus) return;
    const uint32_t nb_cifs = C.geom.nb_cifs;
    DabPlusSubState st = D.st[idx];
    DabPlusEvent* ev = D.events + idx * DP_MAX_EVENTS;
    int32_t n_ev_local = 0;
    uint8_t* sf = D.sf + size_t(s) * (5u * CIF_OUT_STRIDE) + 5u * cfg.out_offset;
    const int n = int(cfg.n_out_bytes);
    for (uint32_t c = 0; c < nb_cifs; c++) {
        if (!C.msc_valid[(size_t(s) * nb_cifs + c) * C.max_subs + sub]) continue;
        const uint8_t* buf = C.msc_out + (size_t(s) * nb_cifs + c) * CIF_OUT_STRIDE + cfg.out_offset;
        dp_process_frame(sh, buf, n, st, sf, D.sf_out + size_t(s) * (5u * CIF_OUT_STRIDE) + 5u * cfg.out_offset, int(5u * cfg.out_offset), ev,
                         &n_ev_local, C.counters, lane);
    }
    if (lane == 0) { D.st[idx] = st; D.n_events[idx] = n_ev_local; }
}

// Persistent CTAs: the field / CRC tables are staged in shared memory once per CTA, then its warps walk the (stream, sub-channel)
// items.  subs_per_stream = largest sub-channel count of the streams in the call (the table has max_subs = 64 rows per stream, a
// full ensemble uses 18: launching a warp per table row spent most of the kernel on CTAs that only loaded the tables).
__global__ void __launch_bounds__(DP_WARPS * 32)
k_dabplus(const ChanDev C, const DabPlusDev D, const int first_stream, const int n_streams, const uint32_t subs_per_stream) {
    __shared__ DpShared sh;
    dp_load_shared(sh);
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t total = uint32_t(n_streams) * subs_per_stream;
    for (uint32_t wid = blockIdx.x * DP_WARPS + (threadIdx.x >> 5); wid < total; wid += gridDim.x * DP_WARPS) {
        const uint32_t si = wid / subs_per_stream, sub = wid - si * subs_per_stream;
        dp_work_item(sh, C, D, uint32_t(first_stream) + si, sub, lane);
        __syncwarp();
    }
}

// Stand-alone AAC_Frame_Processor objects (the C++ adapter of the same name): one warp, one logical frame per call.
struct DabPlusProc {
    DabPlusSubState st;
    int32_t n_events, pad[3];
    DabPlusEvent events[DP_MAX_EVENTS];
    uint8_t sf[5 * CIF_OUT_STRIDE];
    uint8_t sf_out[5 * CIF_OUT_STRIDE];
    uint8_t frame[CIF_OUT_STRIDE];
};

__global__ void __launch_bounds__(32) k_dabplus_direct(DabPlusProc* __restrict__ P, const int n, unsigned long long* __restrict__ counters) {
    __shared__ DpShared sh;
    dp_load_shared(sh);
    const uint32_t lane = threadIdx.x;
    DabPlusSubState st = P->st;
    int32_t n_ev = 0;
    dp_process_frame(sh, P->frame, n, st, P->sf, P->sf_out, 0, P->events, &n_ev, counters, lane);
    if (lane == 0) { P->st = st; P->n_events = n_ev; }
}

// Reed_Solomon_Decoder::Decode batched: one thread per codeword, corrected in place.
__global__ void k_rs_batch(uint8_t* __restrict__ cw, const int n_cw, const int n, const int nroots, const int pad, int* __restrict__ counts,
                           int* __restrict__ positions) {
    __shared__ DpShared sh;
    dp_load_shared(sh);
    const GfTables T{sh.gf_ex, sh.gf_lg};
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_cw) return;
    uint8_t* data = cw + size_t(i) * n;
    uint8_t S[RS_MAX_ROOTS], loc[RS_MAX_ROOTS], xv[RS_MAX_ROOTS], ap[RS_MAX_ROOTS];
    int cnt = 0;
    if (rs_syndromes(T, data, 1, n, nroots, S)) cnt = rs_solve(T, S, nroots, pad, loc, xv, ap);
    for (int j = 0; j < cnt; j++) {
        if (ap[j]) data[int(loc[j]) - pad] ^= xv[j];
        if (positions) positions[size_t(i) * nroots + j] = loc[j];
    }
    counts[i] = cnt;
}

// Packet-mode FEC frame (ETSI EN 300 401 5.3.5; MSC_Reed_Solomon_Data_Packet_Processor::PerformReedSolomonCorrection,
// msc_reed_solomon_data_packet_processor.cpp:200-240): a frame is the 2256-byte application data table followed by the
// 192-byte RS data table, both in transport order.  Because 188 * 12 = 2256 the two tables form ONE column-major 204 x 12
// matrix: byte x of row y sits at x * 12 + y, so the row codewords are stride-12 reads and nothing has to be transposed.
// One thread per (frame, row); a correction is written back only into the application data table (x < 188), like the
// reference, which leaves the FEC packets alone.
#define PKT_FEC_ROWS 12
#define PKT_FEC_DATA 188
#define PKT_FEC_FRAME_BYTES 2448   // 204 * 12
__global__ void k_packet_fec(uint8_t* __restrict__ frames, const int n_frames, int* __restrict__ counts) {
    __shared__ DpShared sh;
    dp_load_shared(sh);
    const GfTables T{sh.gf_ex, sh.gf_lg};
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_frames * PKT_FEC_ROWS) return;
    const int f = i / PKT_FEC_ROWS, y = i - f * PKT_FEC_ROWS;
    uint8_t* row = frames + size_t(f) * PKT_FEC_FRAME_BYTES + y;
    constexpr int nroots = 16, pad = 51, n = 204;
    uint8_t S[RS_MAX_ROOTS], loc[RS_MAX_ROOTS], xv[RS_MAX_ROOTS], ap[RS_MAX_ROOTS];
    int cnt = 0;
    if (rs_syndromes(T, row, PKT_FEC_ROWS, n, nroots, S)) cnt = rs_solve(T, S, nroots, pad, loc, xv, ap);
    for (int j = 0; j < cnt; j++) {
        const int x = int(loc[j]) - pad;
        if (ap[j] && x < PKT_FEC_DATA) row[size_t(x) * PKT_FEC_ROWS] ^= xv[j];
    }
    counts[i] = cnt;
}

static int dabplus_init(DabPlusState& S, int max_streams, int max_subs, int nb_cifs) {
    S.max_streams = max_streams; S.max_subs = max_subs; S.nb_cifs = nb_cifs;
    int rc;
    const size_t n = size_t(max_streams) * max_subs;
    if ((rc = S.d_st.alloc(n * sizeof(DabPlusSubState)))) return rc;
    if ((rc = S.d_sf.alloc(size_t(max_streams) * 5u * CIF_OUT_STRIDE))) return rc;
    if ((rc = S.d_sf_out.alloc(size_t(max_streams) * 5u * CIF_OUT_STRIDE))) return rc;
    if ((rc = S.d_events.alloc(n * DP_MAX_EVENTS * sizeof(DabPlusEvent)))) return rc;
    if ((rc = S.d_nevents.alloc(n * 4))) return rc;
    cudaMemset(S.d_st.p, 0, S.d_st.bytes);
    cudaMemset(S.d_sf.p, 0, S.d_sf.bytes);
    cudaMemset(S.d_sf_out.p, 0, S.d_sf_out.bytes);
    cudaMemset(S.d_events.p, 0, S.d_events.bytes);
    cudaMemset(S.d_nevents.p, 0, S.d_nevents.bytes);
    S.dev.st = S.d_st.as<DabPlusSubState>();
    S.dev.sf = S.d_sf.as<uint8_t>();
    S.dev.sf_out = S.d_sf_out.as<uint8_t>();
    S.dev.events = S.d_events.as<DabPlusEvent>();
    S.dev.n_events = S.d_nevents.as<int32_t>();
    return DABGPU_OK;
}

static void dabplus_destroy(DabPlusState& S) {
    DevBuf* bufs[] = {&S.d_st, &S.d_sf, &S.d_sf_out, &S.d_events, &S.d_nevents, &S.d_rs_cw, &S.d_rs_cnt, &S.d_rs_pos};
    for (DevBuf* b : bufs) b->release();
}

static int dabplus_reset_stream(DabPlusState& S, int stream) {
    CUDA_TRY(cudaMemset(S.dev.st + size_t(stream) * S.max_subs, 0, size_t(S.max_subs) * sizeof(DabPlusSubState)));
    CUDA_TRY(cudaMemset(S.dev.n_events + size_t(stream) * S.max_subs, 0, size_t(S.max_subs) * 4));
    return DABGPU_OK;
}

static int dabplus_run(DabPlusState& S, const ChanDev& C, int first, int n, uint32_t subs_per_stream, int num_sms, cudaStream_t stream, uint64_t* launches,
                       Profiler& pf) {
    if (subs_per_stream == 0) return DABGPU_OK;
    const uint32_t warps = uint32_t(n) * subs_per_stream;
    const uint32_t ctas = std::min((warps + DP_WARPS - 1) / DP_WARPS, uint32_t(num_sms) * 8u);
    pf.begin(PROF_DABPLUS, stream);
    k_dabplus<<<ctas, DP_WARPS * 32, 0, stream>>>(C, S.dev, first, n, subs_per_stream);
    pf.end(stream);
    (*launches)++;
    CUDA_TRY(cudaGetLastError());
    return DABGPU_OK;
}

// Host side: rebuild the flat observer log (same layout as oracle/ref_harness.cpp) from the device records.
static int dabplus_get_events(DabPlusState& S, int stream, int sub, uint8_t* log_host, size_t log_cap, size_t* log_bytes) {
    const size_t idx = size_t(stream) * S.max_subs + sub;
    int32_t n_ev = 0;
    CUDA_TRY(cudaMemcpy(&n_ev, S.dev.n_events + idx, 4, cudaMemcpyDeviceToHost));
    if (n_ev > DP_MAX_EVENTS) return set_error(DABGPU_ERR_OVERFLOW, "event queue overflow (%d events)", n_ev);
    DabPlusEvent ev[DP_MAX_EVENTS];
    if (n_ev > 0) CUDA_TRY(cudaMemcpy(ev, S.dev.events + idx * DP_MAX_EVENTS, size_t(n_ev) * sizeof(DabPlusEvent), cudaMemcpyDeviceToHost));
    size_t off = 0;
    std::vector<uint8_t> sfbuf;
    for (int i = 0; i < n_ev; i++) {
        const size_t padded = (size_t(ev[i].payload_len) + 3u) & ~size_t(3);
        if (off + 24 + padded > log_cap) return set_error(DABGPU_ERR_OVERFLOW, "event log buffer too small");
        const int32_t hdr[6] = {ev[i].type, ev[i].a, ev[i].b, ev[i].c, ev[i].d, ev[i].payload_len};
        memcpy(log_host + off, hdr, 24);
        off += 24;
        if (ev[i].payload_len > 0) {
            // payloads (access units) live in the corrected superframe buffer of the sub-channel
            if (sfbuf.empty()) {
                sfbuf.resize(5u * CIF_OUT_STRIDE);
                CUDA_TRY(cudaMemcpy(sfbuf.data(), S.dev.sf_out + size_t(stream) * (5u * CIF_OUT_STRIDE), sfbuf.size(), cudaMemcpyDeviceToHost));
            }
            memset(log_host + off, 0, padded);
            // payload_off is an offset inside the stream's superframe arena
            memcpy(log_host + off, sfbuf.data() + size_t(ev[i].payload_off), size_t(ev[i].payload_len));
            off += padded;
        }
    }
    if (log_bytes) *log_bytes = off;
    return DABGPU_OK;
}

static int dabplus_rs_decode_batch(DabPlusState& S, uint8_t* cw_host, int n_cw, int nroots, int pad, int* counts_host, int* pos_host,
                                   cudaStream_t stream, uint64_t* launches) {
    if (n_cw <= 0) return DABGPU_OK;
    if (nroots < 1 || nroots > RS_MAX_ROOTS) return set_error(DABGPU_ERR_INVALID, "nroots %d out of range", nroots);
    if (pad < 0 || pad >= 255 - nroots) return set_error(DABGPU_ERR_INVALID, "pad %d out of range", pad);
    const int n = 255 - pad;
    int rc;
    if ((rc = S.d_rs_cw.alloc(size_t(n_cw) * n))) return rc;
    if ((rc = S.d_rs_cnt.alloc(size_t(n_cw) * 4))) return rc;
    if ((rc = S.d_rs_pos.alloc(size_t(n_cw) * nroots * 4))) return rc;
    CUDA_TRY(cudaMemcpyAsync(S.d_rs_cw.p, cw_host, size_t(n_cw) * n, cudaMemcpyHostToDevice, stream));
    CUDA_TRY(cudaMemsetAsync(S.d_rs_pos.p, 0, size_t(n_cw) * nroots * 4, stream));
    k_rs_batch<<<(n_cw + 63) / 64, 64, 0, stream>>>(S.d_rs_cw.as<uint8_t>(), n_cw, n, nroots, pad, S.d_rs_cnt.as<int>(), S.d_rs_pos.as<int>());
    (*launches)++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(cw_host, S.d_rs_cw.p, size_t(n_cw) * n, cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaMemcpyAsync(counts_host, S.d_rs_cnt.p, size_t(n_cw) * 4, cudaMemcpyDeviceToHost, stream));
    if (pos_host) CUDA_TRY(cudaMemcpyAsync(pos_host, S.d_rs_pos.p, size_t(n_cw) * nroots * 4, cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    return DABGPU_OK;
}

static int dabplus_packet_fec_batch(DabPlusState& S, uint8_t* frames_host, int n_frames, int* counts_host, cudaStream_t stream, uint64_t* launches) {
    if (n_frames <= 0) return DABGPU_OK;
    int rc;
    const size_t bytes = size_t(n_frames) * PKT_FEC_FRAME_BYTES, n_rows = size_t(n_frames) * PKT_FEC_ROWS;
    if ((rc = S.d_rs_cw.alloc(bytes))) return rc;
    if ((rc = S.d_rs_cnt.alloc(n_rows * 4))) return rc;
    CUDA_TRY(cudaMemcpyAsync(S.d_rs_cw.p, frames_host, bytes, cudaMemcpyHostToDevice, stream));
    k_packet_fec<<<unsigned((n_rows + 63) / 64), 64, 0, stream>>>(S.d_rs_cw.as<uint8_t>(), n_frames, S.d_rs_cnt.as<int>());
    (*launches)++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(frames_host, S.d_rs_cw.p, bytes, cudaMemcpyDeviceToHost, stream));
    if (counts_host) CUDA_TRY(cudaMemcpyAsync(counts_host, S.d_rs_cnt.p, n_rows * 4, cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    return DABGPU_OK;
}
