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
