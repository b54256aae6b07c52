// ofdm_host.cuh -- host side of the OFDM stage: tables, buffers, launches.
#pragma once
#include "ofdm_demod.cuh"

static int demod_set_attributes(int N, int fmt);

// ---------------------------------------------------------------------------------------------
// Host side
// ---------------------------------------------------------------------------------------------
struct OfdmState {
    uint64_t launches = 0;
    Profiler* prof = nullptr;
    OfdmDev dev;
    dabgpu_params P;
    int max_streams = 0, frame_slots = 0;
    size_t ring_cap = 0;          // internal ring capacity (samples)
    bool external_ring = false;
    int bps = 2;
    DevBuf d_diag, d_diag_meta, d_diag_fft, d_ring, d_st, d_null_ring, d_corr, d_head, d_phase, d_tw, d_prs_conj, d_prs_time, d_dpos, d_outpos, d_obin, d_stage, d_produced;
    int num_sms = 148;
    // k_ofdm_demod2 CTAs per SM are capped (through the shared-memory request) while a channel decode runs on its own stream: its
    // kernels then find room next to the demodulator instead of queueing behind a full wave of it (0 = no cap)
    int demod_ctas_cap = 0;
    // second stream: the streams of a launch are split in two groups so that the latency-bound control kernel of one
    // group overlaps the demodulation kernel of the other
    cudaStream_t aux_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;

    PinnedBuf h_produced;
    std::vector<unsigned long long> h_written;   // absolute samples written per stream (internal ring)
};

// PRS phases, EN 300 401 clause 14.3.2 tables 23/24 (reference: dab_prs_ref.cpp:24-194).
// per block of 32 carriers: (i << 2) | n ; negative carriers first
static const uint8_t kPrsH[4][32] = {
    {0, 2, 0, 0, 0, 0, 1, 1, 2, 0, 0, 0, 2, 2, 1, 1, 0, 2, 0, 0, 0, 0, 1, 1, 2, 0, 0, 0, 2, 2, 1, 1},
    {0, 3, 2, 3, 0, 1, 3, 0, 2, 1, 2, 3, 2, 3, 3, 0, 0, 3, 2, 3, 0, 1, 3, 0, 2, 1, 2, 3, 2, 3, 3, 0},
    {0, 0, 0, 2, 0, 2, 1, 3, 2, 2, 0, 2, 2, 0, 1, 3, 0, 0, 0, 2, 0, 2, 1, 3, 2, 2, 0, 2, 2, 0, 1, 3},
    {0, 1, 2, 1, 0, 3, 3, 2, 2, 3, 2, 1, 2, 1, 3, 2, 0, 1, 2, 1, 0, 3, 3, 2, 2, 3, 2, 1, 2, 1, 3, 2},
};
static const uint8_t kPrsBlocks1[48] = {1, 6, 8, 13, 3, 6, 10, 15, 2, 5, 10, 15, 1, 6, 11, 15, 2, 6, 10, 13, 1, 7, 9, 14,
                                        3, 13, 9, 5, 2, 14, 9, 4, 2, 14, 11, 7, 0, 14, 9, 7, 3, 15, 11, 4, 3, 12, 9, 5};
static const uint8_t kPrsBlocks2[12] = {2, 7, 10, 14, 1, 6, 8, 6, 2, 13, 8, 7};
static const uint8_t kPrsBlocks3[6] = {2, 7, 8, 14, 10, 6};
static const uint8_t kPrsBlocks4[24] = {0, 5, 9, 14, 2, 6, 8, 15, 3, 5, 11, 14, 0, 13, 8, 6, 0, 13, 10, 6, 2, 13, 11, 4};

static void host_prs_spectrum(int mode, int N, int K, std::vector<float2>& prs) {
    const uint8_t* tab = (mode == 1) ? kPrsBlocks1 : (mode == 2) ? kPrsBlocks2 : (mode == 3) ? kPrsBlocks3 : kPrsBlocks4;
    prs.assign(size_t(N), make_float2(0.0f, 0.0f));
    for (int slot = 0; slot < K; slot++) {
        const int k = (slot < K / 2) ? (slot - K / 2) : (slot - K / 2 + 1);
        const int i = tab[slot / 32] >> 2, n = tab[slot / 32] & 3;
        const float phi = float(M_PI) / 2.0f * float(kPrsH[i][slot % 32] + n);
        prs[size_t(k < 0 ? N + k : k)] = make_float2(cosf(phi), sinf(phi));
    }
}

static void host_dft_double(std::vector<double>& re, std::vector<double>& im, bool inverse) {
    // simple recursive-free radix-2 on doubles for table generation only
    const size_t n = re.size();
    for (size_t i = 1, j = 0; i < n; i++) {
        size_t bit = n >> 1;
        for (; j & bit; bit >>= 1) j ^= bit;
        j ^= bit;
        if (i < j) { std::swap(re[i], re[j]); std::swap(im[i], im[j]); }
    }
    for (size_t len = 2; len <= n; len <<= 1) {
        const double ang = (inverse ? 2.0 : -2.0) * M_PI / double(len);
        for (size_t i = 0; i < n; i += len)
            for (size_t k = 0; k < len / 2; k++) {
                const double wr = cos(ang * double(k)), wi = sin(ang * double(k));
                const double ur = re[i + k], ui = im[i + k];
                const double vr = re[i + k + len / 2] * wr - im[i + k + len / 2] * wi;
                const double vi = re[i + k + len / 2] * wi + im[i + k + len / 2] * wr;
                re[i + k] = ur + vr; im[i + k] = ui + vi;
                re[i + k + len / 2] = ur - vr; im[i + k + len / 2] = ui - vi;
            }
    }
}

static int ofdm_init(OfdmState& O, const dabgpu_config& cfg, const dabgpu_params& P, int frame_slots, int8_t* d_frames,
                     uint32_t* d_frames_written, dabgpu_frame_info* d_frame_info, unsigned long long* d_counters) {
    O.P = P;
    O.max_streams = cfg.max_streams;
    O.frame_slots = frame_slots;
    O.bps = (cfg.iq_format == DABGPU_IQ_U8) ? 2 : 8;
    const int S = cfg.max_streams, N = P.nb_fft, K = P.nb_data_carriers;
    size_t cap = cfg.ring_samples;
    if (cap == 0) {
        cap = 1;
        // four frames: room for one pipelined step being copied in while the previous one is demodulated (dabgpu_submit)
        while (cap < size_t(P.nb_frame_samples) * 4 + size_t(P.nb_null_period + P.nb_symbol_period)) cap <<= 1;
    }
    if (cap & (cap - 1)) return set_error(DABGPU_ERR_INVALID, "ring_samples must be a power of two");
    if (cap < size_t(P.nb_frame_samples) + size_t(P.nb_null_period + P.nb_symbol_period) + 4096)
        return set_error(DABGPU_ERR_INVALID, "ring_samples too small for one frame");
    O.ring_cap = cap;
    int rc;
    if ((rc = O.d_ring.alloc(size_t(S) * cap * O.bps))) return rc;
    if ((rc = O.d_st.alloc(size_t(S) * sizeof(OfdmStream)))) return rc;
    if ((rc = O.d_null_ring.alloc(size_t(S) * P.nb_null_period * sizeof(float2)))) return rc;
    if ((rc = O.d_corr.alloc(size_t(S) * (P.nb_null_period + P.nb_symbol_period) * sizeof(float2)))) return rc;
    if ((rc = O.d_head.alloc(size_t(S) * (P.nb_symbol_period + P.nb_cyclic_prefix) * sizeof(float2)))) return rc;
    if ((rc = O.d_phase.alloc(size_t(S) * P.nb_frame_symbols * sizeof(float)))) return rc;
    if (cfg.flags & DABGPU_FLAG_DIAG_TAPS) {
        if ((rc = O.d_diag.alloc(size_t(S) * 2 * size_t(P.nb_fft) * sizeof(float)))) return rc;
        cudaMemset(O.d_diag.p, 0, O.d_diag.bytes);
        if ((rc = O.d_diag_meta.alloc(size_t(S) * sizeof(OfdmDiagMeta)))) return rc;
        cudaMemset(O.d_diag_meta.p, 0, O.d_diag_meta.bytes);
    }
    if ((rc = O.d_produced.alloc(size_t(S)))) return rc;
    if ((rc = O.h_produced.alloc(size_t(S)))) return rc;
    cudaMemset(O.d_ring.p, 0, O.d_ring.bytes);
    cudaMemset(O.d_st.p, 0, O.d_st.bytes);
    cudaMemset(O.d_null_ring.p, 0, O.d_null_ring.bytes);   // the reference's joint block is zero initialised (joint_allocate.h:21-23)
    cudaMemset(O.d_corr.p, 0, O.d_corr.bytes);
    cudaMemset(O.d_head.p, 0, O.d_head.bytes);
    cudaMemset(O.d_phase.p, 0, O.d_phase.bytes);
    O.h_written.assign(size_t(S), 0ull);

    // tables
    std::vector<float2> tw(static_cast<size_t>(N)), prs;
    for (int n = 0; n < N; n++) {
        const double a = -2.0 * M_PI * double(n) / double(N);
        tw[size_t(n)] = make_float2(float(cos(a)), float(sin(a)));
    }
    host_prs_spectrum(cfg.transmission_mode, N, K, prs);
    std::vector<float2> prs_conj(static_cast<size_t>(N)), prs_time(static_cast<size_t>(N));
    for (int i = 0; i < N; i++) prs_conj[size_t(i)] = make_float2(prs[size_t(i)].x, -prs[size_t(i)].y);
    {
        // conj(IFFT(conj(X[i]) * X[i+1]))   (ofdm_demodulator.cpp:136-140)
        std::vector<double> re(static_cast<size_t>(N), 0.0), im(static_cast<size_t>(N), 0.0);
        for (int i = 0; i < N - 1; i++) {
            const double ar = prs[size_t(i)].x, ai = prs[size_t(i)].y, br = prs[size_t(i + 1)].x, bi = prs[size_t(i + 1)].y;
            re[size_t(i)] = ar * br + ai * bi;
            im[size_t(i)] = ar * bi - ai * br;
        }
        host_dft_double(re, im, true);
        for (int i = 0; i < N; i++) prs_time[size_t(i)] = make_float2(float(re[size_t(i)]), float(-im[size_t(i)]));
    }
    // digit reversal of the in-place DIF (radices 8,8,8,4 / 8,8,8,2 / 8,8,8 / 8,8,4)
    std::vector<int> radices;
    switch (N) {
    case 2048: radices = {8, 8, 8, 4}; break;
    case 1024: radices = {8, 8, 8, 2}; break;
    case 512: radices = {8, 8, 8}; break;
    default: radices = {8, 8, 4}; break;
    }
    std::vector<uint16_t> dpos(static_cast<size_t>(N)), outpos(static_cast<size_t>(K));
    for (int k = 0; k < N; k++) {
        int a = 0, rem = N, kk = k;
        for (int R : radices) { const int d = kk % R; kk /= R; rem /= R; a += d * rem; }
        dpos[size_t(k)] = uint16_t(OFDM_PAD(a));
    }
    {
        // frequency de-interleaver (dab_mapper_ref.cpp:10-50) composed with the carrier -> FFT bin map (ofdm_demodulator.cpp:853-864)
        std::vector<int> cmap;
        int v = 0;
        const int dc = N / 2, lo = dc - K / 2, hi = dc + K / 2;
        for (int i = 0; i < N; i++) {
            if (i > 0) v = (13 * v + N / 4 - 1) % N;
            if (v < lo || v > hi || v == dc) continue;
            cmap.push_back(v < dc ? v - lo : v - lo - 1);
        }
        for (int i = 0; i < K; i++) {
            const int slot = cmap[size_t(i)];
            const int kf = (slot < K / 2) ? (slot - K / 2) : (slot - K / 2 + 1);
            outpos[size_t(i)] = dpos[size_t((N + kf) % N)];
        }
    }
    // demod kernel (ofdm_demod.cuh): DIF radices {4|2|1},8,8,8 -- position a = sum k_i * M_i holds bin k = k_1 + R_1 k_2 + ...
    std::vector<uint16_t> obin(static_cast<size_t>(N), uint16_t(0xFFFF));
    {
        std::vector<int> rad2;
        switch (N) {
        case 2048: rad2 = {4, 8, 8, 8}; break;
        case 1024: rad2 = {2, 8, 8, 8}; break;
        case 512: rad2 = {8, 8, 8}; break;
        default: rad2 = {4, 8, 8}; break;
        }
        std::vector<int> cmap;
        int v = 0;
        const int dc = N / 2, lo = dc - K / 2, hi = dc + K / 2;
        for (int i = 0; i < N; i++) {
            if (i > 0) v = (13 * v + N / 4 - 1) % N;
            if (v < lo || v > hi || v == dc) continue;
            cmap.push_back(v < dc ? v - lo : v - lo - 1);
        }
        for (int i = 0; i < K; i++) {
            const int slot = cmap[size_t(i)];
            const int kf = (slot < K / 2) ? (slot - K / 2) : (slot - K / 2 + 1);
            int kk = (N + kf) % N, a = 0, rem = N;
            for (int R : rad2) { const int d = kk % R; kk /= R; rem /= R; a += d * rem; }
            obin[size_t(a)] = uint16_t(i);
        }
    }
    if ((rc = O.d_obin.alloc(obin.size() * 2))) return rc;
    cudaMemcpy(O.d_obin.p, obin.data(), obin.size() * 2, cudaMemcpyHostToDevice);
    if ((rc = O.d_tw.alloc(tw.size() * sizeof(float2)))) return rc;
    if ((rc = O.d_prs_conj.alloc(prs_conj.size() * sizeof(float2)))) return rc;
    if ((rc = O.d_prs_time.alloc(prs_time.size() * sizeof(float2)))) return rc;
    if ((rc = O.d_dpos.alloc(dpos.size() * 2))) return rc;
    if ((rc = O.d_outpos.alloc(outpos.size() * 2))) return rc;
    cudaMemcpy(O.d_tw.p, tw.data(), tw.size() * sizeof(float2), cudaMemcpyHostToDevice);
    cudaMemcpy(O.d_prs_conj.p, prs_conj.data(), prs_conj.size() * sizeof(float2), cudaMemcpyHostToDevice);
    cudaMemcpy(O.d_prs_time.p, prs_time.data(), prs_time.size() * sizeof(float2), cudaMemcpyHostToDevice);
    cudaMemcpy(O.d_dpos.p, dpos.data(), dpos.size() * 2, cudaMemcpyHostToDevice);
    cudaMemcpy(O.d_outpos.p, outpos.data(), outpos.size() * 2, cudaMemcpyHostToDevice);

    OfdmDev& D = O.dev;
    D.g.L = P.nb_frame_symbols; D.g.Tsym = P.nb_symbol_period; D.g.Tnull = P.nb_null_period; D.g.CP = P.nb_cyclic_prefix;
    D.g.N = N; D.g.K = K; D.g.frame_bits = P.nb_frame_bits; D.g.frame_samples = P.nb_frame_samples;
    D.g.sym_per_chunk = (P.nb_frame_symbols == 153) ? 19 : 15;
    D.g.n_chunks = (P.nb_frame_symbols - 1 + D.g.sym_per_chunk - 1) / D.g.sym_per_chunk;
    D.cfg = cfg.ofdm;
    D.iq_format = cfg.iq_format;
    D.ring = O.d_ring.as<uint8_t>();
    D.ring_stride = cap;
    D.ring_mask = cap - 1;
    D.st = O.d_st.as<OfdmStream>();
    D.null_ring = O.d_null_ring.as<float2>();
    D.corr = O.d_corr.as<float2>();
    D.head = O.d_head.as<float2>();
    D.phase_err = O.d_phase.as<float>();
    D.diag = O.d_diag.as<float>();   // null unless DABGPU_FLAG_DIAG_TAPS
    D.diag_meta = O.d_diag_meta.as<OfdmDiagMeta>();
    D.tw = O.d_tw.as<float2>();
    D.prs_fft_conj = O.d_prs_conj.as<float2>();
    D.prs_time_ref = O.d_prs_time.as<float2>();
    D.dpos = O.d_dpos.as<uint16_t>();
    D.outpos = O.d_outpos.as<uint16_t>();
    D.obin = O.d_obin.as<uint16_t>();
    D.tma_ok = 1;   // internal ring: cudaMalloc base, power-of-two capacity
    {
        int dev_id = 0, sms = 148;
        cudaGetDevice(&dev_id);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev_id);
        O.num_sms = sms;
    }
    if ((rc = demod_set_attributes(N, cfg.iq_format))) return rc;
    CUDA_TRY(cudaStreamCreateWithFlags(&O.aux_stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreateWithFlags(&O.ev_fork, cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&O.ev_join, cudaEventDisableTiming));
    D.frames = d_frames;
    D.frames_written = d_frames_written;
    D.frame_info = d_frame_info;
    D.slot_mask = uint32_t(frame_slots - 1);
    D.counters = d_counters;
    D.fg.nb_cifs = uint32_t(P.nb_cifs);
    D.fg.cif_shift = (P.nb_cifs == 4) ? 2u : (P.nb_cifs == 2 ? 1u : 0u);
    D.fg.frame_bits = uint32_t(P.nb_frame_bits);
    D.fg.fic_bits = uint32_t(P.nb_fic_bits);
    D.fg.cif_bits = uint32_t(P.nb_cif_bits);
    D.fg.slot_mask = uint32_t(frame_slots - 1);
    return DABGPU_OK;
}

static void ofdm_destroy(OfdmState& O) {
    DevBuf* bufs[] = {&O.d_diag, &O.d_diag_meta, &O.d_diag_fft, &O.d_ring, &O.d_st, &O.d_null_ring, &O.d_corr, &O.d_head, &O.d_phase, &O.d_tw, &O.d_prs_conj, &O.d_prs_time,
                      &O.d_dpos, &O.d_outpos, &O.d_obin, &O.d_stage, &O.d_produced};
    for (DevBuf* b : bufs) b->release();
    if (O.aux_stream) { cudaStreamSynchronize(O.aux_stream); cudaStreamDestroy(O.aux_stream); O.aux_stream = nullptr; }
    if (O.ev_fork) cudaEventDestroy(O.ev_fork);
    if (O.ev_join) cudaEventDestroy(O.ev_join);
    O.ev_fork = O.ev_join = nullptr;
    O.h_produced.release();
}

static int ofdm_reset(OfdmState& O, int stream, cudaStream_t cs) {
    const int n = (stream < 0) ? O.max_streams : 1;
    k_ofdm_reset<<<(n + 127) / 128, 128, 0, cs>>>(O.dev, stream, n, 0);
    O.launches++;
    CUDA_TRY(cudaGetLastError());
    return DABGPU_OK;
}

// At most n CTAs of k_ofdm_demod2 per SM (by asking for 1/n of the shared memory).  DABGPU_DEMOD_CTAS overrides (tuning knob).
static int demod_smem_request(int need, int cap) {
    if (const char* e = getenv("DABGPU_DEMOD_CTAS")) cap = atoi(e);
    if (cap >= 1 && cap <= 8) return std::max(need, (227 * 1024) / cap - 2048);
    return need;
}

template <int N, int FMT> static int demod_set_attr_t() {
    CUDA_TRY(cudaFuncSetAttribute(k_ofdm_demod2<N, FMT>, cudaFuncAttributeMaxDynamicSharedMemorySize, std::max(int(DemodCfg<N, FMT>::SMEM), 227 * 1024 - 2048)));
    return DABGPU_OK;
}
static int demod_set_attributes(int N, int fmt) {
    const bool u8 = fmt == DABGPU_IQ_U8;
    switch (N) {
    case 2048: return u8 ? demod_set_attr_t<2048, DABGPU_IQ_U8>() : demod_set_attr_t<2048, DABGPU_IQ_C32>();
    case 1024: return u8 ? demod_set_attr_t<1024, DABGPU_IQ_U8>() : demod_set_attr_t<1024, DABGPU_IQ_C32>();
    case 512: return u8 ? demod_set_attr_t<512, DABGPU_IQ_U8>() : demod_set_attr_t<512, DABGPU_IQ_C32>();
    case 256: return u8 ? demod_set_attr_t<256, DABGPU_IQ_U8>() : demod_set_attr_t<256, DABGPU_IQ_C32>();
    }
    return set_error(DABGPU_ERR_INVALID, "unsupported FFT size %d", N);
}

// Symbols per CTA.  A chunk of c symbols costs c+1 FFTs (the first spectrum is only the DQPSK reference), so fewer, longer
// chunks waste less; but every SM should end up with the same number of CTAs.  Model fitted to a sweep on B200 (256
// streams, 4 resident CTAs per SM: 19 symbols per chunk was fastest, then 15, 13, 10, 25, 38): the busiest SM runs
// ceil(ctas / SMs) CTAs of (spc + 1) symbols each, and k co-resident CTAs deliver perf(k) times the throughput of one.
static int demod_pick_chunk(const OfdmState& O, int n, int ctas_per_sm) {
    static const double perf[5] = {1.0, 1.0, 1.9, 2.6, 3.0};
    const int rows = O.P.nb_frame_symbols - 1;
    int best_spc = rows;
    double best = 1e30;
    for (int chunks = 1; chunks <= 16; chunks++) {
        const int spc = (rows + chunks - 1) / chunks;
        const int nch = (rows + spc - 1) / spc;
        const long ctas = long(n) * nch;
        const long per_sm = (ctas + O.num_sms - 1) / O.num_sms;
        const int k = int(per_sm < ctas_per_sm ? per_sm : ctas_per_sm);
        const double cost = double(spc + 1) * double(per_sm) / perf[k > 4 ? 4 : k];
        if (cost < best - 1e-9) { best = cost; best_spc = spc; }
    }
    return best_spc;
}

template <int N, int FMT>
static void ofdm_launch_group(OfdmState& O, int first, int n, int n_samples, int block_size, int max_frames, cudaStream_t cs) {
    const int ctas_per_sm = (N == 2048) ? 4 : (N == 1024 ? 6 : 8);
    int spc = demod_pick_chunk(O, n, ctas_per_sm);
    if (const char* e = getenv("DABGPU_DEMOD_SPC")) { const int v = atoi(e); if (v >= 1 && v < O.P.nb_frame_symbols) spc = v; }   // tuning knob
    const int n_chunks = (O.P.nb_frame_symbols - 1 + spc - 1) / spc;
    const dim3 dgrid(n_chunks, n);
    Profiler& pf = *O.prof;
    for (int it = 0; it < max_frames; it++) {
        pf.begin(PROF_OFDM_CTL, cs);
        k_ofdm_ctl<N><<<n, N / 8, 0, cs>>>(O.dev, first, n_samples, block_size, it == 0 ? 1 : 0);
        pf.end(cs);
        pf.begin(PROF_OFDM_DEMOD, cs);
        k_ofdm_demod2<N, FMT><<<dgrid, N / 8, demod_smem_request(int(DemodCfg<N, FMT>::SMEM), (N == 2048 && n >= 128) ? O.demod_ctas_cap : 0), cs>>>(O.dev, first, spc);
        pf.end(cs);
        O.launches += 2;
    }
    pf.begin(PROF_OFDM_CTL, cs);
    k_ofdm_ctl<N><<<n, N / 8, 0, cs>>>(O.dev, first, n_samples, block_size, 0);
    pf.end(cs);
    O.launches++;
}

template <int N, int FMT>
static int ofdm_run_t(OfdmState& O, int first, int n, int n_samples, int block_size, cudaStream_t cs) {
    // a frame consumes at least frame_samples - CP new samples (fine time offset >= -CP), so at most this many complete
    const int max_frames = n_samples / (O.P.nb_frame_samples - O.P.nb_cyclic_prefix) + 1;
    // One group on the caller's stream is the default.  The control kernel is latency bound (about 45 us per launch whether it
    // walks 128 or 256 streams), so splitting the streams into two groups on two CUDA streams pays its latency twice: measured
    // 0.420 ms per 256-stream step against 0.399 ms unsplit, and 0.480 ms with the control kernels on high-priority streams
    // and the second group started one kernel late (profiles/README.md, r1f).  DABGPU_OVERLAP_GROUPS=1 keeps the split for
    // experiments.
    const bool split = n >= 64 && !O.prof->on && O.aux_stream != nullptr && getenv("DABGPU_OVERLAP_GROUPS") != nullptr;
    if (!split) {
        ofdm_launch_group<N, FMT>(O, first, n, n_samples, block_size, max_frames, cs);
    } else {
        const int n0 = n / 2;
        CUDA_TRY(cudaEventRecord(O.ev_fork, cs));
        CUDA_TRY(cudaStreamWaitEvent(O.aux_stream, O.ev_fork, 0));
        ofdm_launch_group<N, FMT>(O, first, n0, n_samples, block_size, max_frames, cs);
        ofdm_launch_group<N, FMT>(O, first + n0, n - n0, n_samples, block_size, max_frames, O.aux_stream);
        CUDA_TRY(cudaEventRecord(O.ev_join, O.aux_stream));
        CUDA_TRY(cudaStreamWaitEvent(cs, O.ev_join, 0));
    }
    CUDA_TRY(cudaGetLastError());
    return DABGPU_OK;
}

static int ofdm_run(OfdmState& O, int first, int n, int n_samples, int block_size, cudaStream_t cs) {
    if (n == 0 || n_samples == 0) return DABGPU_OK;
    const bool u8 = O.dev.iq_format == DABGPU_IQ_U8;
    switch (O.P.nb_fft) {
    case 2048: return u8 ? ofdm_run_t<2048, DABGPU_IQ_U8>(O, first, n, n_samples, block_size, cs) : ofdm_run_t<2048, DABGPU_IQ_C32>(O, first, n, n_samples, block_size, cs);
    case 1024: return u8 ? ofdm_run_t<1024, DABGPU_IQ_U8>(O, first, n, n_samples, block_size, cs) : ofdm_run_t<1024, DABGPU_IQ_C32>(O, first, n, n_samples, block_size, cs);
    case 512: return u8 ? ofdm_run_t<512, DABGPU_IQ_U8>(O, first, n, n_samples, block_size, cs) : ofdm_run_t<512, DABGPU_IQ_C32>(O, first, n, n_samples, block_size, cs);
    case 256: return u8 ? ofdm_run_t<256, DABGPU_IQ_U8>(O, first, n, n_samples, block_size, cs) : ofdm_run_t<256, DABGPU_IQ_C32>(O, first, n, n_samples, block_size, cs);
    }
    return set_error(DABGPU_ERR_INVALID, "unsupported FFT size %d", O.P.nb_fft);
}

// Host -> ring copy of `len` samples per stream (source sample offset `done`).  Streams that share the same write
// position go out as one strided 2-D copy (two when the ring wraps); otherwise one copy per stream.
static int ofdm_upload(OfdmState& O, const void* iq_host, size_t stride_bytes, int first, int n, size_t done, size_t len, cudaStream_t cs) {
    const uint8_t* src = static_cast<const uint8_t*>(iq_host);
    bool same = true;
    for (int i = 1; i < n; i++) same = same && (O.h_written[size_t(first + i)] == O.h_written[size_t(first)]);
    if (same && n > 1) {
        unsigned long long w = O.h_written[size_t(first)];
        size_t left = len, off = 0;
        while (left > 0) {
            const size_t pos = size_t(w & (O.ring_cap - 1));
            const size_t run = std::min(left, O.ring_cap - pos);
            CUDA_TRY(cudaMemcpy2DAsync(O.d_ring.as<uint8_t>() + (size_t(first) * O.ring_cap + pos) * O.bps, O.ring_cap * O.bps,
                                       src + (done + off) * O.bps, stride_bytes, run * O.bps, size_t(n), cudaMemcpyHostToDevice, cs));
            w += run; off += run; left -= run;
        }
        for (int i = 0; i < n; i++) O.h_written[size_t(first + i)] = w;
        return DABGPU_OK;
    }
    for (int i = 0; i < n; i++) {
        const int s = first + i;
        unsigned long long w = O.h_written[size_t(s)];
        size_t left = len, off = 0;
        while (left > 0) {
            const size_t pos = size_t(w & (O.ring_cap - 1));
            const size_t run = std::min(left, O.ring_cap - pos);
            CUDA_TRY(cudaMemcpyAsync(O.d_ring.as<uint8_t>() + (size_t(s) * O.ring_cap + pos) * O.bps,
                                     src + size_t(i) * stride_bytes + (done + off) * O.bps, run * O.bps, cudaMemcpyHostToDevice, cs));
            w += run; off += run; left -= run;
        }
        O.h_written[size_t(s)] = w;
    }
    return DABGPU_OK;
}

// samples that may be written ahead of the consumer without touching the frame being assembled or the correlation window
static size_t ofdm_ring_headroom(const dabgpu_params& P, size_t ring_cap) {
    return ring_cap - size_t(P.nb_frame_samples) - size_t(P.nb_null_period + P.nb_symbol_period) - 1024;
}
static size_t ofdm_ring_headroom(const OfdmState& O) { return ofdm_ring_headroom(O.P, O.ring_cap); }

static int ofdm_process(OfdmState& O, const void* iq_host, size_t stride_bytes, int first, int n, int n_samples, int block_size, cudaStream_t cs) {
    if (O.external_ring) return set_error(DABGPU_ERR_STATE, "a device input buffer is attached: use dabgpu_ofdm_advance");
    // the ring must keep the frame being assembled plus the correlation window: bound the samples per pass
    const size_t max_chunk = ofdm_ring_headroom(O);
    const int bs = block_size > 0 ? block_size : n_samples;
    size_t chunk_max = (max_chunk / size_t(bs)) * size_t(bs);   // keep Process() block boundaries intact
    if (chunk_max == 0) return set_error(DABGPU_ERR_INVALID, "block_size %d does not fit the IQ ring (%zu samples)", bs, O.ring_cap);
    for (size_t done = 0; done < size_t(n_samples);) {
        const size_t len = std::min(chunk_max, size_t(n_samples) - done);
        int rc = ofdm_upload(O, iq_host, stride_bytes, first, n, done, len, cs);
        if (rc) return rc;
        rc = ofdm_run(O, first, n, int(len), bs, cs);
        if (rc) return rc;
        done += len;
    }
    CUDA_TRY(cudaStreamSynchronize(cs));
    return DABGPU_OK;
}

static int ofdm_attach(OfdmState& O, const void* d_iq, size_t stride_samples, size_t capacity, cudaStream_t cs) {
    CUDA_TRY(cudaStreamSynchronize(cs));
    O.dev.ring = static_cast<const uint8_t*>(d_iq);
    O.dev.ring_stride = stride_samples;
    O.dev.ring_mask = (capacity & (capacity - 1)) == 0 ? (unsigned long long)(capacity - 1) : ~0ull;
    O.external_ring = true;
    // TMA bulk copies move whole 16-byte blocks: they must never leave the caller's buffer
    O.dev.tma_ok = ((reinterpret_cast<uintptr_t>(d_iq) & 15u) == 0 && (stride_samples * size_t(O.bps)) % 16 == 0 && (capacity * size_t(O.bps)) % 16 == 0) ? 1 : 0;
    k_ofdm_reset<<<(O.max_streams + 127) / 128, 128, 0, cs>>>(O.dev, -1, O.max_streams, 1);
    O.launches++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(cs));
    return DABGPU_OK;
}

static int ofdm_advance(OfdmState& O, int first, int n, int n_samples, int block_size, cudaStream_t cs) {
    if (!O.external_ring) return set_error(DABGPU_ERR_STATE, "no device input attached: use dabgpu_ofdm_process");
    if (n_samples < 0) return set_error(DABGPU_ERR_INVALID, "negative sample count");
    return ofdm_run(O, first, n, n_samples, block_size > 0 ? block_size : n_samples, cs);
}

static int ofdm_get_status(OfdmState& O, int stream, dabgpu_ofdm_status* out, cudaStream_t cs) {
    CUDA_TRY(cudaStreamSynchronize(cs));
    OfdmStream st;
    CUDA_TRY(cudaMemcpy(&st, O.dev.st + stream, sizeof(st), cudaMemcpyDeviceToHost));
    out->state = st.state;
    out->total_frames_read = st.frames_read;
    out->total_frames_desync = st.frames_desync;
    out->fine_time_offset = st.fine_time_offset;
    out->signal_l1_average = st.l1_avg;
    out->freq_coarse_offset = st.coarse;
    out->freq_fine_offset = st.fine;
    out->frames_queued = 0;
    return DABGPU_OK;
}

// GetFrameFFT tap: (L [+1]) x N complex spectra of the last emitted frame of one stream (with_null: plus the NULL-symbol row);
// GetFrameDataVec tap: (L-1) x K DQPSK vectors of the same frame.  DABGPU_ERR_STATE when no frame was emitted yet or the frame
// was not contiguous in the ring (the first frame after an acquisition).
static int ofdm_frame_fft(OfdmState& O, int stream, float* host_fft, bool with_null, float* host_vec, cudaStream_t cs) {
    if (!O.d_diag_meta.p) return set_error(DABGPU_ERR_STATE, "context was created without DABGPU_FLAG_DIAG_TAPS");
    const int L = O.P.nb_frame_symbols, N = O.P.nb_fft, K = O.P.nb_data_carriers;
    int rc;
    if ((rc = O.d_diag_fft.alloc((size_t(L + 1) * N + size_t(L - 1) * K) * sizeof(float2)))) return rc;
    CUDA_TRY(cudaStreamSynchronize(cs));
    OfdmDiagMeta m;
    CUDA_TRY(cudaMemcpy(&m, O.d_diag_meta.as<OfdmDiagMeta>() + stream, sizeof(m), cudaMemcpyDeviceToHost));
    if (!m.valid) return set_error(DABGPU_ERR_STATE, "no frame spectrum available for stream %d yet", stream);
    float2* out = O.d_diag_fft.as<float2>();
    float2* vec = out + size_t(L + 1) * N;
    const int rows = L + 1;
    switch (N) {
    case 2048: k_ofdm_diag_fft<2048><<<rows, 256, 0, cs>>>(O.dev, stream, out); break;
    case 1024: k_ofdm_diag_fft<1024><<<rows, 128, 0, cs>>>(O.dev, stream, out); break;
    case 512: k_ofdm_diag_fft<512><<<rows, 64, 0, cs>>>(O.dev, stream, out); break;
    default: k_ofdm_diag_fft<256><<<rows, 32, 0, cs>>>(O.dev, stream, out); break;
    }
    O.launches++;
    if (host_vec) {
        k_ofdm_diag_dqpsk<<<L - 1, 256, 0, cs>>>(out, vec, N, K);
        O.launches++;
    }
    CUDA_TRY(cudaGetLastError());
    if (host_fft) CUDA_TRY(cudaMemcpyAsync(host_fft, out, size_t(with_null ? L + 1 : L) * N * sizeof(float2), cudaMemcpyDeviceToHost, cs));
    if (host_vec) CUDA_TRY(cudaMemcpyAsync(host_vec, vec, size_t(L - 1) * K * sizeof(float2), cudaMemcpyDeviceToHost, cs));
    CUDA_TRY(cudaStreamSynchronize(cs));
    return DABGPU_OK;
}

// packs the newest frame of every stream that produced one during the last run into (stage, produced) on the device
static int ofdm_gather_latest(OfdmState& O, int first, int n, int8_t* d_stage, uint8_t* d_produced, cudaStream_t cs) {
    const dim3 grid(32, n);
    k_ofdm_gather_latest<<<grid, 256, 0, cs>>>(O.dev, first, d_stage, d_produced);
    O.launches++;
    CUDA_TRY(cudaGetLastError());
    return DABGPU_OK;
}

// the same for the streams whose frame counter moved past d_written0 (a device copy of frames_written[first, first + n))
static int ofdm_gather_since(OfdmState& O, int first, int n, const uint32_t* d_written0, int8_t* d_stage, uint8_t* d_produced, cudaStream_t cs) {
    const dim3 grid(32, n);
    k_ofdm_gather_since<<<grid, 256, 0, cs>>>(O.dev, first, d_written0, d_stage, d_produced);
    O.launches++;
    CUDA_TRY(cudaGetLastError());
    return DABGPU_OK;
}

static int ofdm_fetch_latest(OfdmState& O, int first, int n, int8_t* frames_host, uint8_t* produced, cudaStream_t cs) {
    int rc;
    const size_t fb = size_t(O.P.nb_frame_bits);
    if ((rc = O.d_stage.alloc(size_t(n) * fb))) return rc;
    if ((rc = ofdm_gather_latest(O, first, n, O.d_stage.as<int8_t>(), O.d_produced.as<uint8_t>(), cs))) return rc;
    CUDA_TRY(cudaMemcpyAsync(frames_host, O.d_stage.p, size_t(n) * fb, cudaMemcpyDeviceToHost, cs));
    CUDA_TRY(cudaMemcpyAsync(O.h_produced.p, O.d_produced.p, size_t(n), cudaMemcpyDeviceToHost, cs));
    CUDA_TRY(cudaStreamSynchronize(cs));
    memcpy(produced, O.h_produced.p, size_t(n));
    return DABGPU_OK;
}
