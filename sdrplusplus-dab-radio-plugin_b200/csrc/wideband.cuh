// wideband.cuh -- wideband front end: one overlap-save filter bank per capture that mixes, low-pass filters and decimates every
// ensemble in it to its own 2.048 MS/s c32 stream (dabgpu_wideband_*, include/dabgpu.h).  Replaces the plugin's per-ensemble VFO
// and the reference's examples/apply_frequency_shift.
//
// fs = D x 2.048 MHz.  Block b of a source is the N = 512 D input samples [448 D b - 64 D, 448 D b + 448 D); the filter has
// 64 D + 1 taps, so the last 448 D samples of the block's circular convolution are valid, i.e. outputs 448 b .. 448 b + 447 after
// decimation by D.  The N-point forward FFT of a block (bin spacing fs / N = 4 kHz for every D) is shared by all channels of the
// source.  Channel k takes the 512 bins b_k + u, u in [-256, 256), b_k = f^_k / 4 kHz, multiplies them by H[u] (the N-point DFT
// of the taps, / N) and by the block's mixing phase exp(-j 2 pi b_k (448 D b - 64 D) / N) = exp(-j 2 pi b_k (7 b - 1) / 8), and a
// 512-point inverse FFT gives the decimated outputs (the first 64 are the overlap and are dropped).  Keeping 512 of the N bins is
// the decimation: what it drops lies beyond 1.024 MHz, >= 75 dB down.  The residual offset delta_k = f_k - f^_k is a rotation
// of each output sample, its phase formed from the absolute sample index modulo fs in integers.
//
// One CTA of 64 D threads per (block, source): fft_cta<N> forward, then D groups of 64 threads run fft_cta<512> inverse for one
// channel each, as many rounds as the source has channels per group.
#pragma once
#include "ofdm.cuh"

#define WB_OUT 448        // new output samples per block and channel
#define WB_IFFT 512       // inverse FFT points per channel (4 kHz bins at 2.048 MS/s)
#define WB_GROUP 64       // threads of one channel's inverse FFT (fft_cta runs N / 8 threads)

struct WbChan {
    int bin;     // b_k: f^_k / 4000
    int delta;   // f_k - f^_k, Hz
    int out;     // output stream (= channel index)
    int pad;
};

struct WbDev {
    const uint8_t* ring;            // raw input, source s sample a at ring + ((s << ring_log2) + (a & ring_mask)) * bytes/sample
    int ring_log2;
    unsigned long long ring_mask;
    float2* out;                    // channel c sample n at out[c * out_cap + (n & (out_cap - 1))]
    unsigned long long out_cap;
    const float2* H;                // [512] H[u mod 512] / N
    const float2* tw_fwd;           // exp(-j 2 pi k / N), k < N / 8
    const float2* tw_inv;           // exp(-j 2 pi k / 512), k < 64
    const uint16_t* dpos_fwd;       // natural bin -> padded position of the digit-reversed forward output
    const uint16_t* dpos_inv;
    const WbChan* chans;            // channels grouped by source
    const int* chan_first;          // [n_sources + 1]
    long long fs;
};

template <int FMT> struct WbFmt;
template <> struct WbFmt<DABGPU_WB_RAW_U8> {
    static constexpr int BPS = 2;
    __device__ static float2 load(const uint8_t* p) {
        const uchar2 v = *reinterpret_cast<const uchar2*>(p);
        return make_float2((float(v.x) - 127.5f) * (1.0f / 127.5f), (float(v.y) - 127.5f) * (1.0f / 127.5f));
    }
};
template <> struct WbFmt<DABGPU_WB_RAW_S8> {
    static constexpr int BPS = 2;
    __device__ static float2 load(const uint8_t* p) {
        const char2 v = *reinterpret_cast<const char2*>(p);
        return make_float2(float(v.x) * (1.0f / 127.0f), float(v.y) * (1.0f / 127.0f));
    }
};
template <> struct WbFmt<DABGPU_WB_RAW_S16L> {
    static constexpr int BPS = 4;
    __device__ static float2 load(const uint8_t* p) {
        const short2 v = *reinterpret_cast<const short2*>(p);
        return make_float2(float(v.x) * (1.0f / 32767.0f), float(v.y) * (1.0f / 32767.0f));
    }
};
template <> struct WbFmt<DABGPU_WB_RAW_F32L> {
    static constexpr int BPS = 8;
    __device__ static float2 load(const uint8_t* p) { return *reinterpret_cast<const float2*>(p); }
};

template <int D> struct WbCfg {
    static constexpr int N = 512 * D, NT = N / 8;
    static constexpr int SMEM = (2 * OFDM_PAD(N) + D * 2 * OFDM_PAD(WB_IFFT)) * int(sizeof(float));
};

// grid = (blocks, sources), block = 64 D threads; blocks block0 .. block0 + gridDim.x - 1.  1 024 threads per SM (64 registers):
// at 98 registers a D = 8 CTA would run alone on its SM
template <int D, int FMT>
__global__ void __launch_bounds__(64 * D, 16 / D) k_wideband(const WbDev W, const unsigned long long block0) {
    constexpr int N = WbCfg<D>::N, NT = WbCfg<D>::NT;
    extern __shared__ float wb_smem[];
    float* f_re = wb_smem;
    float* f_im = wb_smem + OFDM_PAD(N);
    const int tid = threadIdx.x, s = blockIdx.y;
    const unsigned long long b = block0 + blockIdx.x;

    // forward FFT of the block, input before sample 0 counts as zero
    {
        const long long a0 = (long long)(b * (WB_OUT * D)) - 64LL * D;
        const uint8_t* src = W.ring + (size_t(s) << W.ring_log2) * WbFmt<FMT>::BPS;
        float2 x[8];
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const long long a = a0 + tid + j * NT;
            x[j] = a < 0 ? make_float2(0.0f, 0.0f) : WbFmt<FMT>::load(src + size_t((unsigned long long)a & W.ring_mask) * WbFmt<FMT>::BPS);
        }
        fft_cta<N, false>(x, f_re, f_im, W.tw_fwd, tid);
    }

    const int g = tid / WB_GROUP, lt = tid % WB_GROUP;
    float* g_re = wb_smem + 2 * OFDM_PAD(N) + g * 2 * OFDM_PAD(WB_IFFT);
    float* g_im = g_re + OFDM_PAD(WB_IFFT);
    const int c0 = W.chan_first[s], nch = W.chan_first[s + 1] - c0;
    const int bphase = int((7ull * b + 7ull) & 7ull);   // (7 b - 1) mod 8
    // (448 D b) mod fs: start of the block's outputs on the input clock
    const long long t0 = (long long)((b * (unsigned long long)(WB_OUT * D)) % (unsigned long long)W.fs);
    for (int r = 0; r * D < nch; r++) {
        __syncthreads();   // forward spectrum complete / previous round's outputs read
        const int c = r * D + g;
        const bool active = c < nch;
        WbChan ch = {0, 0, 0, 0};
        float2 y[8];
        if (active) {
            ch = W.chans[c0 + c];
            const int p = ((ch.bin & 7) * bphase) & 7;
            float sn, cs;
            sincospif(-0.25f * float(p), &sn, &cs);
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int i = lt + j * WB_GROUP;
                const int u = i < WB_IFFT / 2 ? i : i - WB_IFFT;
                const int pos = W.dpos_fwd[(ch.bin + u) & (N - 1)];
                const float2 h = cmulf(__ldg(W.H + i), make_float2(cs, sn));
                y[j] = cmulf(make_float2(f_re[pos], f_im[pos]), h);
            }
        } else {
#pragma unroll
            for (int j = 0; j < 8; j++) y[j] = make_float2(0.0f, 0.0f);
        }
        fft_cta<WB_IFFT, true>(y, g_re, g_im, W.tw_inv, lt);
        __syncthreads();
        if (active) {
            float2* dst = W.out + size_t(ch.out) * W.out_cap;
#pragma unroll
            for (int j = 0; j < WB_OUT / WB_GROUP; j++) {
                const int m = lt + j * WB_GROUP;
                const int pos = W.dpos_inv[64 + m];
                float2 v = make_float2(g_re[pos], g_im[pos]);
                if (ch.delta != 0) {
                    long long t = t0 + m * D;   // (n D) mod fs, n = 448 b + m
                    if (t >= W.fs) t -= W.fs;
                    long long ph = (t * ch.delta) % W.fs;
                    if (ph < 0) ph += W.fs;
                    float sn, cs;
                    sincospif(-2.0f * (float(ph) / float(W.fs)), &sn, &cs);
                    v = cmulf(v, make_float2(cs, sn));
                }
                dst[(b * WB_OUT + m) & (W.out_cap - 1)] = v;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Any rate the plan supports (dabgpu_wideband_plan): the same overlap-save filter bank with a forward FFT of N_in = fs / bin_hz
// points (a product of 2, 3 and 5, <= 8192) and NOUT = 2.048 MHz / bin_hz bins kept per channel.  Block b of a source is the
// N_in input samples [step_in b - ov_in, step_in b + step_in), ov_in = N_in - step_in; its NOUT-point inverse FFT gives outputs at
// input times a0 + n' fs / 2.048 MHz, of which the last step_out are kept: outputs step_out b .. step_out b + step_out - 1.  The
// bin index of a channel wraps modulo N_in, its mixing phase is exp(-j 2 pi ((b_k a0) mod N_in) / N_in) and the residual
// rotation of output n is exp(-j 2 pi ((n delta) mod 2 048 000) / 2 048 000), all from exact integers.
//
// One CTA of WB_MIX_THREADS threads per (block, source): an in-place mixed-radix DIF FFT of the block in shared memory (pass
// radices from the host, 8s first, then 4 or 2, then 3s, then 5s; output digit reversed, dpos_fwd maps a natural bin to its
// position), then WB_MIX_THREADS / (NOUT / 8) groups run fft_cta<NOUT> inverse for one channel each.
// ---------------------------------------------------------------------------------------------
#define WB_MIX_THREADS 256
#define WB_MIX_MAX_FFT 8192
#define WB_MIX_MAX_PASSES 14   // 8192 = 8^4 x 2 needs 5, 6561 = 3^8 needs 8

struct WbMixDev {
    WbDev w;                        // H: [NOUT] H[u mod NOUT] / N_in; tw_fwd: exp(-j 2 pi k / N_in), k < N_in; tw_inv, dpos_inv: NOUT
    int n_fft, step_in, ov_in, step_out;
    int n_pass;
    int radix[WB_MIX_MAX_PASSES];
};

template <int NOUT> struct WbMixCfg {
    static constexpr int GT = NOUT / 8, G = WB_MIX_THREADS / GT;
    static constexpr int GROUP_FLOATS = G * 2 * OFDM_PAD(NOUT);
    static constexpr int SMEM_MAX = (2 * OFDM_PAD(WB_MIX_MAX_FFT) + GROUP_FLOATS) * int(sizeof(float));
};

__device__ __forceinline__ void dft3f(float2& a0, float2& a1, float2& a2) {
    const float s = 0.86602540378443864676f;
    const float2 t = make_float2(a1.x + a2.x, a1.y + a2.y), d = make_float2(s * (a1.x - a2.x), s * (a1.y - a2.y));
    const float2 m = make_float2(a0.x - 0.5f * t.x, a0.y - 0.5f * t.y);
    a0 = make_float2(a0.x + t.x, a0.y + t.y);
    a1 = make_float2(m.x + d.y, m.y - d.x);   // m - j d
    a2 = make_float2(m.x - d.y, m.y + d.x);
}

__device__ __forceinline__ void dft5f(float2& a0, float2& a1, float2& a2, float2& a3, float2& a4) {
    const float c1 = 0.30901699437494742410f, c2 = -0.80901699437494742410f;
    const float s1 = 0.95105651629515357212f, s2 = 0.58778525229247312917f;
    const float2 t1 = make_float2(a1.x + a4.x, a1.y + a4.y), t2 = make_float2(a2.x + a3.x, a2.y + a3.y);
    const float2 d1 = make_float2(a1.x - a4.x, a1.y - a4.y), d2 = make_float2(a2.x - a3.x, a2.y - a3.y);
    const float2 A1 = make_float2(a0.x + c1 * t1.x + c2 * t2.x, a0.y + c1 * t1.y + c2 * t2.y);
    const float2 A2 = make_float2(a0.x + c2 * t1.x + c1 * t2.x, a0.y + c2 * t1.y + c1 * t2.y);
    const float2 B1 = make_float2(s1 * d1.x + s2 * d2.x, s1 * d1.y + s2 * d2.y);
    const float2 B2 = make_float2(s2 * d1.x - s1 * d2.x, s2 * d1.y - s1 * d2.y);
    a0 = make_float2(a0.x + t1.x + t2.x, a0.y + t1.y + t2.y);
    a1 = make_float2(A1.x + B1.y, A1.y - B1.x);   // A1 - j B1
    a4 = make_float2(A1.x - B1.y, A1.y + B1.x);
    a2 = make_float2(A2.x + B2.y, A2.y - B2.x);
    a3 = make_float2(A2.x - B2.y, A2.y + B2.x);
}

// in-place forward DIF FFT of n points at re/im (padded), every thread of the CTA
__device__ __forceinline__ void fft_mixed_fwd(float* __restrict__ re, float* __restrict__ im, const WbMixDev& W, const int tid) {
    const int n = W.n_fft;
    int M = n;
    for (int p = 0; p < W.n_pass; p++) {
        const int R = W.radix[p], m = M / R, tstride = n / M;
        __syncthreads();
        for (int t = tid; t < n / R; t += WB_MIX_THREADS) {
            const int q = t / m, r = t - q * m, base = q * M + r;
            float2 y[8];
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int a = OFDM_PAD(base + j * m);
                y[j] = j < R ? make_float2(re[a], im[a]) : make_float2(0.0f, 0.0f);
            }
            switch (R) {
            case 8: dft8<false>(y); break;
            case 4: dft4<false>(y[0], y[1], y[2], y[3]); break;
            case 2: { const float2 u = y[0]; y[0] = make_float2(u.x + y[1].x, u.y + y[1].y); y[1] = make_float2(u.x - y[1].x, u.y - y[1].y); } break;
            case 3: dft3f(y[0], y[1], y[2]); break;
            default: dft5f(y[0], y[1], y[2], y[3], y[4]); break;
            }
            float2 wp[8];
            if (m > 1) tw_powers7(__ldg(W.w.tw_fwd + r * tstride), wp);
#pragma unroll
            for (int k = 0; k < 8; k++) {
                if (k >= R) break;
                float2 v = y[k];
                if (k > 0 && m > 1) v = cmulf(v, wp[k]);
                const int a = OFDM_PAD(base + k * m);
                re[a] = v.x; im[a] = v.y;
            }
        }
        M = m;
    }
}

// grid = (blocks, sources), block = WB_MIX_THREADS; blocks block0 .. block0 + gridDim.x - 1.  64 registers: 4 CTAs of
// different sources share an SM where shared memory allows (3 at N_in = 5000)
template <int NOUT, int FMT>
__global__ void __launch_bounds__(WB_MIX_THREADS, 4) k_wideband_mixed(const WbMixDev W, const unsigned long long block0) {
    constexpr int GT = WbMixCfg<NOUT>::GT;
    const int n = W.n_fft;
    extern __shared__ float wb_smem[];
    float* f_re = wb_smem;
    float* f_im = wb_smem + OFDM_PAD(n);
    const int tid = threadIdx.x, s = blockIdx.y;
    const unsigned long long b = block0 + blockIdx.x;
    const long long a0 = (long long)(b * (unsigned long long)W.step_in) - W.ov_in;

    // block input, converted, in natural order; input before sample 0 counts as zero
    {
        const uint8_t* src = W.w.ring + (size_t(s) << W.w.ring_log2) * WbFmt<FMT>::BPS;
        for (int i = tid; i < n; i += WB_MIX_THREADS) {
            const long long a = a0 + i;
            const float2 x = a < 0 ? make_float2(0.0f, 0.0f) : WbFmt<FMT>::load(src + size_t((unsigned long long)a & W.w.ring_mask) * WbFmt<FMT>::BPS);
            f_re[OFDM_PAD(i)] = x.x; f_im[OFDM_PAD(i)] = x.y;
        }
    }
    fft_mixed_fwd(f_re, f_im, W, tid);

    const int g = tid / GT, lt = tid % GT;
    float* g_re = wb_smem + 2 * OFDM_PAD(n) + g * 2 * OFDM_PAD(NOUT);
    float* g_im = g_re + OFDM_PAD(NOUT);
    const int c0 = W.w.chan_first[s], nch = W.w.chan_first[s + 1] - c0;
    const long long a0m = ((a0 % n) + n) % n;
    // (step_out b) mod 2 048 000: the block's first output on the 2.048 MHz clock
    const long long t0 = (long long)((b * (unsigned long long)W.step_out) % 2048000ull);
    const int drop = NOUT - W.step_out;
    for (int r = 0; r * WbMixCfg<NOUT>::G < nch; r++) {
        __syncthreads();   // forward spectrum complete / previous round's outputs read
        const int c = r * WbMixCfg<NOUT>::G + g;
        const bool active = c < nch;
        WbChan ch = {0, 0, 0, 0};
        float2 y[8];
        if (active) {
            ch = W.w.chans[c0 + c];
            const int bm = ch.bin < 0 ? ch.bin + n : ch.bin;
            const int p = int((long long)bm * a0m % n);
            float sn, cs;
            sincospif(-2.0f * (float(p) / float(n)), &sn, &cs);
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int i = lt + j * GT;
                int k = ch.bin + (i < NOUT / 2 ? i : i - NOUT);   // |k| < n: the channel lies within +-fs/2
                k += k < 0 ? n : 0;
                k -= k >= n ? n : 0;
                const int pos = W.w.dpos_fwd[k];
                const float2 h = cmulf(__ldg(W.w.H + i), make_float2(cs, sn));
                y[j] = cmulf(make_float2(f_re[pos], f_im[pos]), h);
            }
        } else {
#pragma unroll
            for (int j = 0; j < 8; j++) y[j] = make_float2(0.0f, 0.0f);
        }
        fft_cta<NOUT, true>(y, g_re, g_im, W.w.tw_inv, lt);
        __syncthreads();
        if (active) {
            float2* dst = W.w.out + size_t(ch.out) * W.w.out_cap;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int m = lt + j * GT;
                if (m >= W.step_out) break;
                const int pos = W.w.dpos_inv[drop + m];
                float2 v = make_float2(g_re[pos], g_im[pos]);
                if (ch.delta != 0) {
                    long long t = t0 + m;   // n mod 2 048 000, n = step_out b + m
                    if (t >= 2048000) t -= 2048000;
                    long long ph = (t * ch.delta) % 2048000;
                    if (ph < 0) ph += 2048000;
                    float sn, cs;
                    sincospif(-2.0f * (float(ph) / 2048000.0f), &sn, &cs);
                    v = cmulf(v, make_float2(cs, sn));
                }
                dst[(b * (unsigned long long)W.step_out + m) & (W.w.out_cap - 1)] = v;
            }
        }
    }
}
