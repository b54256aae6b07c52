// ofdm.cuh -- batched OFDM demodulator: per-stream control kernel (sync state machine) + wide
// frame demodulation kernel (PLL -> cyclic-prefix phase -> FFT -> DQPSK -> frequency de-interleave
// -> int8 soft bits in one pass over the IQ).
//
// Reference (paths relative to /root/reference/vendor/DAB-Radio/src/ofdm):
//   OFDM_Demod::Process and its five states            ofdm_demodulator.cpp:235-577
//   CoordinatorThread / PipelineThread                 ofdm_demodulator.cpp:581-766
//   CalculateCyclicPhaseError / fine frequency update  ofdm_demodulator.cpp:768-840
//   CalculateDQPSK / CalculateViterbiBits              ofdm_demodulator.cpp:842-889, 58-72
//   apply_pll_avx + chebyshev sine                     dsp/apply_pll.cpp:82-116, dsp/chebyshev_sine.h:13-105
//   complex_conj_mul_sum                               dsp/complex_conj_mul_sum.cpp:65-99
//   CircularBuffer / ReconstructionBuffer / frame buf  circular_buffer.h, reconstruction_buffer.h, ofdm_frame_buffer.h
//   tables                                             dab_prs_ref.cpp:24-194, dab_mapper_ref.cpp:10-50
//
// Ordering is the canonical serialised one (SURVEY.md appendix C): when a frame completes, the control
// kernel stops consuming samples of that stream, the demod kernel processes the frame, and the next
// control pass applies the fine-frequency update before the next frame's PRS is looked at.
//
// Layout: the raw IQ of every stream stays where the host (or the caller's device buffer) put it, in a
// ring addressed by absolute sample index; frames are never copied, the demod kernel reads the ring
// directly (2 B/sample for u8 input) and writes only the 1 B/bit soft decisions.  The first symbol of a
// frame comes from a small per-stream "head" buffer because the reference takes it from its correlation
// buffer (which, while acquiring, is not always contiguous with the stream: circular_buffer.h quirk).
#pragma once
#include "common.cuh"
#include "viterbi.cuh"   // GatherGeom / frame_convert_group: layout of the soft-bit frame ring

enum { OST_FINDING_NULL = 0, OST_READING_NULL_PRS = 1, OST_COARSE = 2, OST_FINE_TIME = 3, OST_READING_SYMBOLS = 4 };

#define OFDM_PAD(a) ((a) + (((a) >> 5) << 2))
#define OFDM_L1_BATCH 512

struct OfdmStream {
    int32_t state, frames_read, frames_desync, coarse_found;
    float coarse, fine;
    int32_t fine_time_offset, null_start_found, null_end_found;
    float l1_avg;
    uint32_t ring_index, ring_len, corr_len;
    uint32_t frame_fill, n_head;
    int32_t pending;          // 1 = a complete frame waits for / is being processed by k_ofdm_demod
    float frame_f;            // coarse+fine sampled when the frame was handed over (ofdm_demodulator.cpp:672)
    int32_t block_size;
    int32_t produced_last;    // frames emitted during the last process/advance call
    int32_t corr_contig;      // the correlation buffer holds consecutive ring samples ending at `consumed` (steady state)
    int32_t head_contig;      // the frame being assembled is contiguous in the ring from frame_ring_base - n_head
    int32_t pad0;
    unsigned long long consumed, push_end, block_end, frame_ring_base;
};

// Position and frequency of the last frame handed to the observers, kept for the on-demand GetFrameFFT tap.
struct OfdmDiagMeta { unsigned long long abs0; float f; int32_t valid; };

struct OfdmGeom {
    int L, Tsym, Tnull, CP, N, K, frame_bits, frame_samples, sym_per_chunk, n_chunks;
};

struct OfdmDev {
    OfdmGeom g;
    dabgpu_ofdm_config cfg;
    int iq_format;
    // input ring
    const uint8_t* ring;              // base of stream 0
    unsigned long long ring_stride;   // samples between streams
    unsigned long long ring_mask;     // capacity-1 when the capacity is a power of two, else all ones (no wrap)
    // per-stream buffers
    OfdmStream* st;
    float2* null_ring;   // [stream][Tnull]
    float2* corr;        // [stream][Tnull+Tsym]
    float2* head;        // [stream][Tsym+CP]
    float* phase_err;    // [stream][L]
    float* diag;         // optional (DABGPU_FLAG_DIAG_TAPS): [stream][2][N] = impulse response, coarse frequency response (dB)
    struct OfdmDiagMeta* diag_meta;   // optional: where the last emitted frame of every stream sits in the IQ ring
    // tables
    const float2* tw;            // exp(-2*pi*i*n/N)
    const float2* prs_fft_conj;  // conj(PRS spectrum), natural order
    const float2* prs_time_ref;  // conj(IFFT(relative phase of PRS)), natural order
    const uint16_t* dpos;        // padded smem position of natural index k after the in-place DIF FFT
    const uint16_t* outpos;      // padded smem position of the carrier that feeds output bit i (frequency de-interleaver)
    const uint16_t* obin;        // demod kernel: [N] output index (0..K-1) of the bin at FFT-output position a, 0xFFFF = unused bin
    int tma_ok;                  // ring base/stride/capacity are multiples of 16 bytes: TMA bulk staging may be used
    // outputs
    int8_t* frames;              // [stream][slot][frame_bits]
    uint32_t* frames_written;    // [stream]
    dabgpu_frame_info* frame_info;   // [stream][slot]
    uint32_t slot_mask;
    unsigned long long* counters;
    GatherGeom fg;               // frame ring layout (planar MSC, viterbi.cuh)
};

__device__ __forceinline__ float2 cmulf(const float2 a, const float2 b) { return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }

__device__ __forceinline__ float2 ofdm_ring_sample(const OfdmDev& D, const int s, const unsigned long long abs_idx) {
    const unsigned long long off = (unsigned long long)s * D.ring_stride + (abs_idx & D.ring_mask);
    if (D.iq_format == DABGPU_IQ_U8) {
        // QuantisedIQToFloatIQ<uint8_t>: (u8 - 127.5) * (1/127.5)   (app_iq_readers.h:23-43, 72-87)
        const uchar2 v = __ldg(reinterpret_cast<const uchar2*>(D.ring) + off);
        return make_float2(__fmul_rn(__fsub_rn(float(v.x), 127.5f), 1.0f / 127.5f), __fmul_rn(__fsub_rn(float(v.y), 127.5f), 1.0f / 127.5f));
    }
    return __ldg(reinterpret_cast<const float2*>(D.ring) + off);
}

// sin(2*pi*x) on [-0.5, 0.5], same polynomial and (AVX+FMA build) evaluation order as chebyshev_sine.h:79-105
__device__ __forceinline__ float cheb_sin(const float x) {
    const float z = __fmul_rn(x, x);
    float b = 3.20396066f;
    b = __fmaf_rn(b, z, -14.07150173f);
    b = __fmaf_rn(b, z, 38.50016403f);
    b = __fmaf_rn(b, z, -67.07687378f);
    b = __fmaf_rn(b, z, 64.83583069f);
    b = __fmaf_rn(b, z, -25.13274193f);
    return __fmul_rn(__fmul_rn(x, b), __fadd_rn(z, -0.25f));
}

// apply_pll_avx (dsp/apply_pll.cpp:82-116): y = x * exp(j*2*pi*(dt0 + n*f)), float32 phase arithmetic reproduced
// operation by operation: base = fma(float(n & ~3), f, dt0); t = base + (float(n&3)*f [+0.25]); t -= rint(t)
__device__ __forceinline__ float2 pll_rotate(const float2 v, const int n, const float f, const float dt0) {
    const float base = __fmaf_rn(float(n & ~3), f, dt0);
    const float kf = __fmul_rn(float(n & 3), f);
    float ts = __fadd_rn(base, kf);
    float tc = __fadd_rn(base, __fadd_rn(kf, 0.25f));
    ts = __fsub_rn(ts, rintf(ts));
    tc = __fsub_rn(tc, rintf(tc));
    const float sn = cheb_sin(ts), cs = cheb_sin(tc);
    return make_float2(__fmaf_rn(cs, v.x, -__fmul_rn(sn, v.y)), __fmaf_rn(cs, v.y, __fmul_rn(sn, v.x)));
}

// ---------------------------------------------------------------------------------------------
// CTA-wide in-place decimation-in-frequency FFT in shared memory, N/8 threads, radix 8 (+ final 4 or 2).
// Stage-1 inputs come in registers: x[j] = input[tid + j*N/8].  Output is digit reversed; D.dpos maps a
// natural index to its (padded) position.  Arrays are split re/im and padded (OFDM_PAD) so that the
// strided stage accesses hit distinct banks.
// ---------------------------------------------------------------------------------------------
template <bool INV> __device__ __forceinline__ float2 mul_neg_i(const float2 t) {   // t * (-i) forward, t * (+i) inverse
    return INV ? make_float2(-t.y, t.x) : make_float2(t.y, -t.x);
}

template <bool INV> __device__ __forceinline__ void dft4(float2& d0, float2& d1, float2& d2, float2& d3) {
    const float2 s02 = make_float2(d0.x + d2.x, d0.y + d2.y), m02 = make_float2(d0.x - d2.x, d0.y - d2.y);
    const float2 s13 = make_float2(d1.x + d3.x, d1.y + d3.y), m13 = mul_neg_i<INV>(make_float2(d1.x - d3.x, d1.y - d3.y));
    d0 = make_float2(s02.x + s13.x, s02.y + s13.y);
    d2 = make_float2(s02.x - s13.x, s02.y - s13.y);
    d1 = make_float2(m02.x + m13.x, m02.y + m13.y);
    d3 = make_float2(m02.x - m13.x, m02.y - m13.y);
}

template <bool INV> __device__ __forceinline__ void dft8(float2 (&a)[8]) {
    const float h = 0.70710678118654752440f;
    float2 b0 = make_float2(a[0].x + a[4].x, a[0].y + a[4].y), c0 = make_float2(a[0].x - a[4].x, a[0].y - a[4].y);
    float2 b1 = make_float2(a[1].x + a[5].x, a[1].y + a[5].y), c1 = make_float2(a[1].x - a[5].x, a[1].y - a[5].y);
    float2 b2 = make_float2(a[2].x + a[6].x, a[2].y + a[6].y), c2 = make_float2(a[2].x - a[6].x, a[2].y - a[6].y);
    float2 b3 = make_float2(a[3].x + a[7].x, a[3].y + a[7].y), c3 = make_float2(a[3].x - a[7].x, a[3].y - a[7].y);
    // c_j *= w^j, w = exp(-+ 2*pi*i/8)
    if (!INV) {
        c1 = make_float2((c1.x + c1.y) * h, (c1.y - c1.x) * h);
        c2 = make_float2(c2.y, -c2.x);
        c3 = make_float2((c3.y - c3.x) * h, -(c3.x + c3.y) * h);
    } else {
        c1 = make_float2((c1.x - c1.y) * h, (c1.y + c1.x) * h);
        c2 = make_float2(-c2.y, c2.x);
        c3 = make_float2(-(c3.x + c3.y) * h, (c3.x - c3.y) * h);
    }
    dft4<INV>(b0, b1, b2, b3);
    dft4<INV>(c0, c1, c2, c3);
    a[0] = b0; a[2] = b1; a[4] = b2; a[6] = b3;
    a[1] = c0; a[3] = c1; a[5] = c2; a[7] = c3;
}

// w^1 .. w^7 from one table entry.  The twiddles of a pass are powers of one root per thread; fetching them from the table
// cost seven loads with a different 32-byte sector per lane (strides of 32 k bytes): those loads, not arithmetic or barriers, were
// what bounded the kernel -- 1.03 -> 0.73 ms per 1024 frames with six complex multiplies instead.
__device__ __forceinline__ void tw_powers7(const float2 w1, float2 (&w)[8]) {
    w[1] = w1; w[2] = cmulf(w1, w1); w[3] = cmulf(w[2], w1); w[4] = cmulf(w[2], w[2]);
    w[5] = cmulf(w[4], w1); w[6] = cmulf(w[3], w[3]); w[7] = cmulf(w[4], w[3]);
}

template <bool INV> __device__ __forceinline__ float2 ld_tw(const float2* __restrict__ tw, const int idx) {
    float2 w = __ldg(tw + idx);
    if (INV) w.y = -w.y;
    return w;
}

template <int N, bool INV>
__device__ __forceinline__ void fft_cta(float2 (&x)[8], float* __restrict__ re, float* __restrict__ im, const float2* __restrict__ tw, const int tid) {
    constexpr int NT = N / 8;
    dft8<INV>(x);
    {
        float2 wp[8];
        tw_powers7(ld_tw<INV>(tw, tid), wp);
#pragma unroll
        for (int k = 0; k < 8; k++) {
            float2 v = x[k];
            if (k > 0) v = cmulf(v, wp[k]);
            const int a = OFDM_PAD(tid + k * NT);
            re[a] = v.x; im[a] = v.y;
        }
    }
#pragma unroll
    for (int M = N / 8; M >= 8; M /= 8) {
        __syncthreads();
        const int m8 = M / 8;
        const int q = tid / m8, r = tid - q * m8;
        const int base = q * M + r;
        float2 y[8];
#pragma unroll
        for (int j = 0; j < 8; j++) { const int a = OFDM_PAD(base + j * m8); y[j] = make_float2(re[a], im[a]); }
        dft8<INV>(y);
        float2 wp[8];
        if (M > 8) tw_powers7(ld_tw<INV>(tw, r * (N / M)), wp);
#pragma unroll
        for (int k = 0; k < 8; k++) {
            float2 v = y[k];
            if (k > 0 && M > 8) v = cmulf(v, wp[k]);
            const int a = OFDM_PAD(base + k * m8);
            re[a] = v.x; im[a] = v.y;
        }
    }
    constexpr int RF = (N == 2048 || N == 256) ? 4 : ((N == 1024 || N == 8192) ? 2 : 1);   // N / 8^stages
    if (RF == 4) {
        __syncthreads();
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const int g = tid + h * NT;
            float2 d[4];
#pragma unroll
            for (int j = 0; j < 4; j++) { const int a = OFDM_PAD(4 * g + j); d[j] = make_float2(re[a], im[a]); }
            dft4<INV>(d[0], d[1], d[2], d[3]);
#pragma unroll
            for (int j = 0; j < 4; j++) { const int a = OFDM_PAD(4 * g + j); re[a] = d[j].x; im[a] = d[j].y; }
        }
    } else if (RF == 2) {
        __syncthreads();
#pragma unroll
        for (int h = 0; h < 4; h++) {
            const int p = tid + h * NT;
            const int a0 = OFDM_PAD(2 * p), a1 = OFDM_PAD(2 * p + 1);
            const float2 u = make_float2(re[a0], im[a0]), v = make_float2(re[a1], im[a1]);
            re[a0] = u.x + v.x; im[a0] = u.y + v.y;
            re[a1] = u.x - v.x; im[a1] = u.y - v.y;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Frame demodulation kernel.  grid = (chunks, streams), block = N/8 threads.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float2 ofdm_frame_sample(const OfdmDev& D, const int s, const OfdmStream& st, const uint32_t k,
                                                    const float2* __restrict__ head) {
    if (k < st.n_head) return __ldg(head + k);
    return ofdm_ring_sample(D, s, st.frame_ring_base + (k - st.n_head));
}

// ---------------------------------------------------------------------------------------------
// Control kernel: one CTA (N/8 threads) per stream walks the reference state machine over the
// newly available samples; heavy per-frame work is left to k_ofdm_demod.
// ---------------------------------------------------------------------------------------------
struct CtlShared {
    OfdmStream st;
    float l1[OFDM_L1_BATCH];
    float red_v[32];
    int red_i[32];
    float red_s[32];
    int flag;
    int nb_read;
};

__device__ __forceinline__ void ctl_update_fine(OfdmStream& st, const int N, const float delta) {   // ofdm_demodulator.cpp:829-840
    const float wrap = 0.5f * (1.0f / float(N)) * 1.01f;
    st.fine = fmodf(st.fine + delta, wrap);
}

__device__ __forceinline__ void ctl_reset(OfdmStream& st) {   // OFDM_Demod::Reset, ofdm_demodulator.cpp:277-289
    st.state = OST_FINDING_NULL;
    st.corr_len = 0;
    st.frames_desync++;
    st.coarse_found = 0;
    st.coarse = 0.0f;
    st.fine = 0.0f;
    st.fine_time_offset = 0;
    st.corr_contig = 0;
}

// CalculateL1Average (:922-932) for a batch of windows: window w (< nb) covers `count` samples from a0 + w*stride.
// Two adjacent lanes share a window so that a CTA of NT threads has NT/2 windows and all their loads in flight at
// once (the control kernel is latency bound: one dependent global round trip per batch instead of one per window).
template <int NT>
__device__ __forceinline__ void ctl_l1_batch(const OfdmDev& D, const int s, const unsigned long long a0, const int stride, const int count,
                                             const int nb, float* __restrict__ out, const int tid) {
    const int half = (count + 1) >> 1;
    for (int w0 = 0; w0 < nb; w0 += NT / 2) {
        const int w = w0 + (tid >> 1);
        float acc = 0.0f;
        if (w < nb) {
            const int i0 = (tid & 1) * half, i1 = min(count, i0 + half);
            const unsigned long long base = a0 + (unsigned long long)w * (unsigned long long)stride;
            const unsigned long long pos = (base + (unsigned long long)i0) & D.ring_mask;
            if (D.iq_format == DABGPU_IQ_U8 && count == 100 && (D.ring_mask == ~0ull || pos + 50ull <= D.ring_mask + 1ull)) {
                // the default window (signal_l1.nb_samples = 100) on u8 input: the 100 bytes of this lane's half are fetched as 26
                // aligned words that are all in flight at once -- one memory round trip where the sample loop below makes five
                // dependent ones -- and summed in the same order
                const uintptr_t a = reinterpret_cast<uintptr_t>(D.ring) + 2u * ((unsigned long long)s * D.ring_stride + pos);
                const uint32_t* q = reinterpret_cast<const uint32_t*>(a & ~uintptr_t(3));
                const bool odd = (a & 2u) != 0u;
                uint32_t wd[26];
#pragma unroll
                for (int k = 0; k < 25; k++) wd[k] = __ldg(q + k);
                wd[25] = odd ? __ldg(q + 25) : 0u;
#pragma unroll
                for (int k = 0; k < 25; k++) {
                    const uint32_t r = odd ? __funnelshift_r(wd[k], wd[k + 1], 16) : wd[k];
#pragma unroll
                    for (int h2 = 0; h2 < 2; h2++) {
                        const float x = __fmul_rn(__fsub_rn(float((r >> (16 * h2)) & 0xFFu), 127.5f), 1.0f / 127.5f);
                        const float y = __fmul_rn(__fsub_rn(float((r >> (16 * h2 + 8)) & 0xFFu), 127.5f), 1.0f / 127.5f);
                        acc += fabsf(x) + fabsf(y);
                    }
                }
            } else {
#pragma unroll 10
                for (int i = i0; i < i1; i++) {
                    const float2 v = ofdm_ring_sample(D, s, base + i);
                    acc += fabsf(v.x) + fabsf(v.y);
                }
            }
        }
        acc += __shfl_xor_sync(FULL_MASK, acc, 1);
        if (w < nb && (tid & 1) == 0) out[w] = acc / float(count);
    }
}

template <int N>
__global__ void __launch_bounds__(N / 8, (N == 2048) ? 3 : 4)   // 2048: 80 registers, three CTAs (streams) per SM: 0.317 -> 0.283 ms per 1024-stream step; four (64 registers) spill more than they hide (0.284)
k_ofdm_ctl(const OfdmDev D, const int first_stream, const int n_new_samples, const int block_size, const int is_first) {
    constexpr int NT = N / 8;
    constexpr int NP = N + N / 8;
    constexpr int NW = NT / 32;
    __shared__ float a_re[NP], a_im[NP], b_re[NP], b_im[NP];
    __shared__ CtlShared sh;
    const int s = first_stream + blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const OfdmGeom& g = D.g;
    OfdmStream& st = sh.st;
    // the stream record and the frame's cyclic-prefix phase errors come in with one coalesced round trip each (thread 0 alone
    // took a dependent load per field and per symbol while the rest of the CTA waited at the first barrier: a fifth of the kernel)
    static_assert(sizeof(OfdmStream) % 4 == 0 && sizeof(OfdmStream) <= 4 * NT, "stream record is copied one word per thread");
    if (tid < int(sizeof(OfdmStream) / 4)) reinterpret_cast<uint32_t*>(&sh.st)[tid] = reinterpret_cast<const uint32_t*>(D.st + s)[tid];
    for (int l = tid; l < g.L; l += NT) sh.l1[l] = D.phase_err[size_t(s) * g.L + l];   // L <= 153 < OFDM_L1_BATCH
    __syncthreads();
    if (tid == 0) {
        if (is_first) {
            st.push_end += (unsigned long long)n_new_samples;
            st.block_size = block_size > 0 ? block_size : n_new_samples;
            st.produced_last = 0;
        }
        if (st.pending == 1) {
            // coordinator (ofdm_demodulator.cpp:608-635): average CP phase -> fine frequency, then emit the frame
            float total = 0.0f;
            for (int l = 0; l < g.L; l++) total += sh.l1[l];
            const float avg = total / float(g.L);
            const float err = (1.0f / float(N)) * avg / (2.0f * 3.14159265358979323846f);
            ctl_update_fine(st, N, -D.cfg.fine_freq_update_beta * err);
            st.frames_read++;
            const uint32_t w = D.frames_written[s];
            dabgpu_frame_info fi;
            fi.freq_coarse_offset = st.coarse; fi.freq_fine_offset = st.fine; fi.fine_time_offset = st.fine_time_offset; fi.frame_index = int(w);
            D.frame_info[size_t(s) * (D.slot_mask + 1u) + (w & D.slot_mask)] = fi;
            D.frames_written[s] = w + 1u;
            if (D.diag_meta) {
                OfdmDiagMeta m;
                m.abs0 = st.frame_ring_base - st.n_head; m.f = st.frame_f; m.valid = st.head_contig ? 1 : 0;
                D.diag_meta[s] = m;
            }
            st.produced_last++;
            st.pending = 0;
            atomicAdd(&D.counters[0], 1ull);   // CNT_FRAMES_DEMOD
        }
    }
    float2* null_ring = D.null_ring + size_t(s) * g.Tnull;
    float2* corr = D.corr + size_t(s) * (g.Tnull + g.Tsym);
    float2* head = D.head + size_t(s) * (g.Tsym + g.CP);
    const int K1 = D.cfg.signal_l1_nb_samples;

    for (;;) {
        __syncthreads();
        if (st.pending) break;
        if (st.consumed == st.block_end) {
            if (st.consumed == st.push_end) break;
            // start of the next Process() call: UpdateSignalAverage (ofdm_demodulator.cpp:934-950)
            const unsigned long long bstart = st.consumed;
            const unsigned long long remaining = st.push_end - bstart;
            const int blen = int(remaining < (unsigned long long)st.block_size ? remaining : (unsigned long long)st.block_size);
            __syncthreads();
            if (blen >= K1) {
                const int M = blen - K1, Lstep = K1 * D.cfg.signal_l1_nb_decimate;
                const int n_win = (M + Lstep - 1) / Lstep;
                for (int w0 = 0; w0 < n_win; w0 += OFDM_L1_BATCH) {
                    const int nb = min(OFDM_L1_BATCH, n_win - w0);
                    ctl_l1_batch<NT>(D, s, bstart + (unsigned long long)w0 * Lstep, Lstep, K1, nb, sh.l1, tid);
                    __syncthreads();
                    if (tid == 0) {
                        const float beta = D.cfg.signal_l1_update_beta;
                        float a = st.l1_avg;
                        for (int w = 0; w < nb; w++) a = beta * a + (1.0f - beta) * sh.l1[w];
                        st.l1_avg = a;
                    }
                    __syncthreads();
                }
            }
            if (tid == 0) st.block_end = bstart + (unsigned long long)blen;
            __syncthreads();
        }
        const int rem = int(st.block_end - st.consumed);
        const int state = st.state;

        if (state == OST_FINDING_NULL) {
            // FindNullPowerDip (ofdm_demodulator.cpp:291-347)
            const int M = rem - K1;
            const int n_win = M > 0 ? (M + K1 - 1) / K1 : 0;
            const float t0 = st.l1_avg * D.cfg.null_thresh_start, t1 = st.l1_avg * D.cfg.null_thresh_end;
            if (tid == 0) { sh.nb_read = rem; sh.flag = 0; }
            __syncthreads();
            for (int w0 = 0; w0 < n_win; w0 += OFDM_L1_BATCH) {
                const int nb = min(OFDM_L1_BATCH, n_win - w0);
                ctl_l1_batch<NT>(D, s, st.consumed + (unsigned long long)w0 * K1, K1, K1, nb, sh.l1, tid);
                __syncthreads();
                if (tid == 0) {
                    for (int w = 0; w < nb; w++) {
                        if (st.null_start_found) {
                            if (sh.l1[w] > t1) { st.null_end_found = 1; sh.nb_read = (w0 + w) * K1 + K1; sh.flag = 1; break; }
                        } else if (sh.l1[w] < t0) {
                            st.null_start_found = 1;
                        }
                    }
                }
                __syncthreads();
                if (sh.flag) break;
            }
            const int nb_read = sh.nb_read;
            // CircularBuffer::ConsumeBuffer(read_all = true): only the last Tnull samples survive
            const int cap = g.Tnull;
            const int first = nb_read > cap ? nb_read - cap : 0;
            for (int i = first + tid; i < nb_read; i += NT)
                null_ring[(st.ring_index + uint32_t(i)) % uint32_t(cap)] = ofdm_ring_sample(D, s, st.consumed + i);
            __syncthreads();
            if (tid == 0) {
                st.ring_index = (st.ring_index + uint32_t(nb_read)) % uint32_t(cap);
                st.ring_len = min(st.ring_len + uint32_t(nb_read), uint32_t(cap));
                st.consumed += (unsigned long long)nb_read;
            }
            __syncthreads();
            if (st.null_end_found) {
                const uint32_t Lr = st.ring_len, start = st.ring_index;
                for (uint32_t i = tid; i < Lr; i += NT) corr[i] = null_ring[(i + start) % uint32_t(cap)];
                __syncthreads();
                if (tid == 0) {
                    st.null_start_found = 0; st.null_end_found = 0;
                    st.corr_len = Lr; st.ring_len = 0;
                    st.corr_contig = 0;   // CircularBuffer read-out order is not guaranteed to be stream order (circular_buffer.h)
                    st.state = OST_READING_NULL_PRS;
                }
            }
        } else if (state == OST_READING_NULL_PRS) {
            const int cap = g.Tnull + g.Tsym;
            const int need = cap - int(st.corr_len);
            const int take = rem < need ? rem : need;
            for (int i = tid; i < take; i += NT) corr[st.corr_len + i] = ofdm_ring_sample(D, s, st.consumed + i);
            __syncthreads();
            if (tid == 0) {
                st.corr_len += uint32_t(take);
                st.consumed += (unsigned long long)take;
                if (int(st.corr_len) == cap) st.state = OST_COARSE;
            }
        } else if (state == OST_COARSE) {
            // RunCoarseFreqSync (ofdm_demodulator.cpp:360-471)
            if (!D.cfg.is_coarse_freq_correction) {
                if (tid == 0) { st.coarse = 0.0f; st.state = OST_FINE_TIME; }
                continue;
            }
            const float2* prs = corr + g.Tnull;
            float2 x[8];
#pragma unroll
            for (int j = 0; j < 8; j++) x[j] = prs[tid + j * NT];
            fft_cta<N, false>(x, a_re, a_im, D.tw, tid);
            __syncthreads();
#pragma unroll
            for (int j = 0; j < 8; j++) {   // CalculateRelativePhase: conj(X[i]) * X[i+1]
                const int i = tid + j * NT;
                float2 z = make_float2(0.0f, 0.0f);
                if (i < N - 1) {
                    const int p0 = D.dpos[i], p1 = D.dpos[i + 1];
                    const float2 u = make_float2(a_re[p0], a_im[p0]), v = make_float2(a_re[p1], a_im[p1]);
                    z = make_float2(u.x * v.x + u.y * v.y, u.x * v.y - u.y * v.x);
                }
                x[j] = z;
            }
            fft_cta<N, true>(x, b_re, b_im, D.tw, tid);
            __syncthreads();
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int i = tid + j * NT;
                const int p = D.dpos[i];
                x[j] = cmulf(make_float2(b_re[p], b_im[p]), __ldg(D.prs_time_ref + i));
            }
            __syncthreads();
            fft_cta<N, false>(x, a_re, a_im, D.tw, tid);
            __syncthreads();
            // CalculateMagnitude: resp[i] = 20*log10(|F[(i + N/2) % N]|), kept in b_re (natural order, unpadded)
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int i = tid + j * NT;
                const int p = D.dpos[(i + N / 2) % N];
                b_re[i] = 20.0f * log10f(sqrtf(a_re[p] * a_re[p] + a_im[p] * a_im[p]));
                if (D.diag) D.diag[(size_t(s) * 2 + 1) * N + i] = b_re[i];   // OFDM_Demod::GetCoarseFrequencyResponse
            }
            __syncthreads();
            const int Mh = N / 2;
            int maxoff = int(D.cfg.max_coarse_freq_correction_norm * float(N));
            maxoff = max(0, min(maxoff, Mh));
            // first maximum over i in [-maxoff, maxoff] (fft index i+Mh, skipping index N)
            float bv = -INFINITY; int bi = 0x7fffffff;
            for (int i = -maxoff + tid; i <= maxoff; i += NT) {
                const int k = i + Mh;
                if (k == N) continue;
                const float v = b_re[k];
                if (v > bv || (v == bv && i < bi)) { bv = v; bi = i; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float ov = __shfl_xor_sync(FULL_MASK, bv, o);
                const int oi = __shfl_xor_sync(FULL_MASK, bi, o);
                if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
            }
            if (lane == 0) { sh.red_v[warp] = bv; sh.red_i[warp] = bi; }
            __syncthreads();
            if (tid == 0) {
                for (int w = 1; w < NW; w++)
                    if (sh.red_v[w] > bv || (sh.red_v[w] == bv && sh.red_i[w] < bi)) { bv = sh.red_v[w]; bi = sh.red_i[w]; }
                // the reference starts from max_value = resp[-maxoff+Mh], index -maxoff and only replaces on '>'
                int max_index = bi;
                if (!(bv > b_re[-maxoff + Mh])) max_index = -maxoff;
                float mag[3]; int pk[3];
                for (int j = 0; j < 3; j++) {
                    int idx = max_index - 1 + j;
                    idx = max(-maxoff, min(idx, maxoff));
                    int k = idx + Mh;
                    if (k >= N) k = N - 1;
                    mag[j] = powf(10.0f, b_re[k] / 20.0f);
                    pk[j] = k - Mh;
                }
                const float sum = mag[0] + mag[1] + mag[2];
                float lerp = 0.0f;
                for (int j = 0; j < 3; j++) lerp += float(pk[j]) * mag[j] / sum;
                const float predicted = -lerp / float(N);
                const float error = predicted - st.coarse;
                const bool large = fabsf(error) > 1.5f / float(N);
                const float beta = (large || !st.coarse_found) ? 1.0f : D.cfg.coarse_freq_slow_beta;
                const float delta = beta * error;
                st.coarse += delta;
                st.coarse_found = 1;
                ctl_update_fine(st, N, -delta);
                st.state = OST_FINE_TIME;
            }
        } else if (state == OST_FINE_TIME) {
            // RunFineTimeSync (ofdm_demodulator.cpp:473-548)
            const float2* prs = corr + g.Tnull;
            const float f = st.coarse + st.fine;
            float2 x[8];
#pragma unroll
            for (int j = 0; j < 8; j++) { const int n = tid + j * NT; x[j] = pll_rotate(prs[n], n, f, 0.0f); }
            fft_cta<N, false>(x, a_re, a_im, D.tw, tid);
            __syncthreads();
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int i = tid + j * NT;
                const int p = D.dpos[i];
                x[j] = cmulf(make_float2(a_re[p], a_im[p]), __ldg(D.prs_fft_conj + i));
            }
            fft_cta<N, true>(x, b_re, b_im, D.tw, tid);
            __syncthreads();
            // impulse response in dB, natural order in a_re (unpadded)
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int i = tid + j * NT;
                const int p = D.dpos[i];
                a_re[i] = 20.0f * log10f(sqrtf(b_re[p] * b_re[p] + b_im[p] * b_im[p]));
                if (D.diag) D.diag[(size_t(s) * 2 + 0) * N + i] = a_re[i];   // OFDM_Demod::GetImpulseResponse
            }
            __syncthreads();
            const float decay = 1.0f - D.cfg.impulse_peak_distance_probability;
            float bv = -INFINITY; int bi = 0x7fffffff; float sum = 0.0f;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int i = tid + j * NT;
                const float v = a_re[i];
                const float nd = float(abs(g.CP - i)) / float(g.Tsym);
                const float wv = (1.0f - decay * nd) * v;
                sum += v;
                if (wv > bv || (wv == bv && i < bi)) { bv = wv; bi = i; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float ov = __shfl_xor_sync(FULL_MASK, bv, o);
                const int oi = __shfl_xor_sync(FULL_MASK, bi, o);
                sum += __shfl_xor_sync(FULL_MASK, sum, o);
                if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
            }
            if (lane == 0) { sh.red_v[warp] = bv; sh.red_i[warp] = bi; sh.red_s[warp] = sum; }
            __syncthreads();
            if (tid == 0) {
                for (int w = 1; w < NW; w++) {
                    sum += sh.red_s[w];
                    if (sh.red_v[w] > bv || (sh.red_v[w] == bv && sh.red_i[w] < bi)) { bv = sh.red_v[w]; bi = sh.red_i[w]; }
                }
                // sequential scan semantics: starts from (impulse[0], index 0), replaced only by a strictly larger weighted value
                float max_value = a_re[0]; int max_index = 0;
                if (bv > max_value) { max_value = bv; max_index = bi; }
                const float avg = sum / float(N);
                if ((max_value - avg) < D.cfg.impulse_peak_threshold_db) {
                    ctl_reset(st);
                    sh.flag = 0;
                } else {
                    const int offset = max_index - g.CP;
                    st.n_head = uint32_t(g.Tsym - offset);
                    st.fine_time_offset = offset;
                    sh.flag = 1;
                }
            }
            __syncthreads();
            if (sh.flag) {
                const int offset = st.fine_time_offset;
                const int start = g.Tnull + offset;
                for (uint32_t i = tid; i < st.n_head; i += NT) head[i] = corr[start + i];
                __syncthreads();
                if (tid == 0) {
                    st.frame_fill = st.n_head;
                    st.frame_ring_base = st.consumed;
                    st.head_contig = st.corr_contig;
                    st.corr_len = 0;
                    st.state = OST_READING_SYMBOLS;
                }
            }
        } else {   // OST_READING_SYMBOLS (ofdm_demodulator.cpp:550-577): nothing is copied, the frame stays in the ring
            const int need = g.frame_samples - int(st.frame_fill);
            const int take = rem < need ? rem : need;
            if (take == need) {
                // the NULL symbol at the end of the frame seeds the correlation buffer of the next frame
                const unsigned long long null_abs = st.frame_ring_base + (unsigned long long)(g.L * g.Tsym) - st.n_head;
                for (int i = tid; i < g.Tnull; i += NT) corr[i] = ofdm_ring_sample(D, s, null_abs + i);
            }
            __syncthreads();
            if (tid == 0) {
                st.frame_fill += uint32_t(take);
                st.consumed += (unsigned long long)take;
                if (take == need) {
                    st.corr_len = uint32_t(g.Tnull);
                    st.corr_contig = 1;   // NULL symbol taken from the ring right before `consumed`; READ_NULL_PRS appends what follows
                    st.state = OST_READING_NULL_PRS;
                    st.frame_f = st.coarse + st.fine;
                    st.pending = 1;
                }
            }
        }
    }
    __syncthreads();
    if (tid < int(sizeof(OfdmStream) / 4)) reinterpret_cast<uint32_t*>(D.st + s)[tid] = reinterpret_cast<const uint32_t*>(&sh.st)[tid];
}

// Packs the newest frame of every stream that produced one in the last call into a contiguous staging buffer.
__global__ void k_ofdm_gather_latest(const OfdmDev D, const int first_stream, int8_t* __restrict__ stage, uint8_t* __restrict__ produced) {
    const int s = first_stream + blockIdx.y;
    const OfdmStream& st = D.st[s];
    const bool has = st.produced_last > 0;
    if (blockIdx.x == 0 && threadIdx.x == 0) produced[blockIdx.y] = has ? 1 : 0;
    if (!has) return;
    const uint32_t slot = (D.frames_written[s] - 1u) & D.slot_mask;
    const int8_t* src = D.frames + (size_t(s) * (D.slot_mask + 1u) + slot) * D.g.frame_bits;
    int8_t* dst = stage + size_t(blockIdx.y) * D.g.frame_bits;   // natural order, as the observers of On_OFDM_Frame see it
    const uint32_t n16 = uint32_t(D.g.frame_bits) / 16u;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += gridDim.x * blockDim.x) frame_convert_group(src, dst, i, D.fg, false);
}

// The same over a step that spans several runs (produced_last only covers the last one): stream first_stream + y has produced
// when its frame counter moved past written0[y], the counter as it stood before the step's first run.
__global__ void k_ofdm_gather_since(const OfdmDev D, const int first_stream, const uint32_t* __restrict__ written0, int8_t* __restrict__ stage,
                                    uint8_t* __restrict__ produced) {
    const int s = first_stream + blockIdx.y;
    const uint32_t written = D.frames_written[s];
    const bool has = written != written0[blockIdx.y];
    if (blockIdx.x == 0 && threadIdx.x == 0) produced[blockIdx.y] = has ? 1 : 0;
    if (!has) return;
    const uint32_t slot = (written - 1u) & D.slot_mask;
    const int8_t* src = D.frames + (size_t(s) * (D.slot_mask + 1u) + slot) * D.g.frame_bits;
    int8_t* dst = stage + size_t(blockIdx.y) * D.g.frame_bits;
    const uint32_t n16 = uint32_t(D.g.frame_bits) / 16u;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += gridDim.x * blockDim.x) frame_convert_group(src, dst, i, D.fg, false);
}

// OFDM_Demod::GetFrameFFT (ofdm_demodulator.h:135, filled by PipelineThread, ofdm_demodulator.cpp:673-700): the spectra of the
// PRS and the data symbols of the last emitted frame, natural bin order, recomputed on demand from the IQ that is still in the
// ring (the demodulation kernel keeps its spectra in registers).  One CTA per symbol; same PLL and FFT as the control kernel.
// Row L is the spectrum of the first symbol period of the NULL symbol that follows the frame, like the reference's pipeline
// computes it (GetDataSymbol(L) of ofdm_frame_buffer.h is the head of the NULL symbol; TII lives there).
template <int N>
__global__ void __launch_bounds__(N / 8) k_ofdm_diag_fft(const OfdmDev D, const int s, float2* __restrict__ out) {
    constexpr int NT = N / 8;
    constexpr int NP = N + N / 8;
    __shared__ float a_re[NP], a_im[NP];
    const OfdmDiagMeta m = D.diag_meta[s];
    if (!m.valid) return;
    const OfdmGeom& g = D.g;
    const int l = blockIdx.x, tid = threadIdx.x;
    const float dt0 = __fmul_rn(float(l * g.Tsym), m.f);
    float2 x[8];
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const int n = g.CP + tid + j * NT;
        x[j] = pll_rotate(ofdm_ring_sample(D, s, m.abs0 + (unsigned long long)(l * g.Tsym + n)), n, m.f, dt0);
    }
    fft_cta<N, false>(x, a_re, a_im, D.tw, tid);
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const int i = tid + j * NT;
        const int p = D.dpos[i];
        out[size_t(l) * N + i] = make_float2(a_re[p], a_im[p]);
    }
}

// OFDM_Demod::GetFrameDataVec (ofdm_demodulator.h:136; CalculateDQPSK, ofdm_demodulator.cpp:842-865): row i holds
// X_i[k] * conj(X_{i+1}[k]) for the K data carriers k = -K/2 .. K/2 without 0, before the frequency de-interleaver.
__global__ void k_ofdm_diag_dqpsk(const float2* __restrict__ spec, float2* __restrict__ out, const int N, const int K) {
    const int i = blockIdx.x;
    const float2* x0 = spec + size_t(i) * N;
    const float2* x1 = x0 + N;
    for (int c = threadIdx.x; c < K; c += blockDim.x) {
        const int k = (c < K / 2) ? (c - K / 2) : (c - K / 2 + 1);
        const float2 a = x0[(N + k) % N], b = x1[(N + k) % N];
        out[size_t(i) * K + c] = make_float2(a.x * b.x + a.y * b.y, a.y * b.x - a.x * b.y);
    }
}

__global__ void k_ofdm_reset(const OfdmDev D, const int stream, const int n_streams, const int full) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_streams) return;
    const int s = (stream < 0) ? i : stream;
    OfdmStream st = D.st[s];
    if (full) {
        memset(&st, 0, sizeof(st));
    } else {
        ctl_reset(st);
        st.pending = 0;
    }
    D.st[s] = st;
}

