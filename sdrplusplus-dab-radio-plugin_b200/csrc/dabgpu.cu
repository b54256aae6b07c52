// dabgpu.cu -- libdabgpu.so: C ABI (include/dabgpu.h) over the sm_100a kernels.  Unity build.
#include "common.cuh"
#include "tables.cuh"
#include "viterbi.cuh"
#include "viterbi_lanes.cuh"
#include "chan.cuh"
#include "dabplus.cuh"
#include "packet.cuh"
#include "ofdm_host.cuh"
#include "wideband.cuh"
#include "../host/fic_autoconfig.hpp"
#include "../host/capture_formats.hpp"
#include <algorithm>
#include <numeric>

#define DABGPU_VERSION "dabgpu 0.1 (sm_100a)"

struct SubHost {
    dabgpu_subchannel sc;
    int payload = DABGPU_PAYLOAD_STREAM;
    Schedule sched;
    uint32_t n_out_bytes, out_offset;
    bool active = true;   // false: removed by dabgpu_msc_remove_subchannel (the index stays reserved so that the others keep theirs)
    int64_t pkt_region = -1;   // packet entries: offset of their region in the packet pool
    uint64_t pkt_cap = 0;      // ... and its log capacity (pkt_item_bound)
    bool is_packet() const { return payload == DABGPU_PAYLOAD_PACKET || payload == DABGPU_PAYLOAD_PACKET_FEC; }
};

struct dabgpu_ctx {
    dabgpu_config cfg;
    dabgpu_params P;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int num_sms = 0;
    uint64_t launches = 0;
    int frame_slots = 0, max_subs = 0;
    Profiler prof;

    // Viterbi
    DevBuf d_prbs, d_counter, d_scratch, d_jobs;
    uint32_t scratch_steps = 0;
    int vit_blocks = 0;
    size_t prbs_words = 0;
    DevBuf d_vsoft, d_vout, d_verr;   // staging of dabgpu_viterbi_decode
    // lane-per-trellis batch path (viterbi_lanes.cuh)
    DevBuf d_vlplan, d_vllist, d_vlsym, d_vlscratch;
    int vl_mode = 0;                  // 0 auto, 1 always, 2 never
    uint32_t vl_min_jobs = 6144;      // auto: lanes from this many active trellises per call
    uint32_t vl_scratch_slots = 0;    // decoder warps the decision scratch is sized for
    int vl_ctas_forced = 0;           // test hook: 1 or 4 CTAs per SM regardless of the call size
    uint32_t vl_scratch_rows = 0;
    struct { int first = -1, n = -1; uint64_t epoch = 0; uint32_t count[VL_BUCKETS]; uint32_t max_steps = 0; uint32_t max_subs_used = 0; } vl_cache;
    uint64_t cfg_epoch = 1;

    // soft-bit frame ring + channel decode state
    DevBuf d_frames, d_frames_written, d_frames_decoded, d_frame_info;
    DevBuf d_pushstage, d_popstage;   // natural-order frames on their way into / out of the ring (dabgpu_softbits_push, dabgpu_ofdm_pop_frames)
    DevBuf d_frames_snapshot;   // frames_written as the channel decode sees it (copied on the main stream before the fork)
    DevBuf d_subcfg, d_nsubs, d_cifs_consumed;
    DevBuf d_fic_out, d_fic_crc, d_msc_out, d_msc_valid, d_status, d_counters;
    DevBuf d_deint;   // de-interleaved CIFs of the frame being decoded (k_chan_deinterleave)
    std::vector<std::vector<SubHost>> subs;
    ChanDev chan;
    PinnedBuf h_status, h_stage;
    std::vector<uint32_t> h_frames_popped;   // per stream, host side cursor of dabgpu_ofdm_pop_frames
    std::vector<uint32_t> h_frames_dropped;  // per stream, frames dabgpu_ofdm_pop_frames could not deliver (overwritten in the ring)

    // DAB+ superframe stage
    DabPlusState dabplus;
    // packet-mode sub-channels
    PacketState packet;
    // channel stream: dabgpu_chan_decode runs on it (see there); join_dabplus() makes the main stream wait for it
    cudaStream_t s_dp = nullptr;
    cudaEvent_t ev_dp = nullptr, ev_dp_fork = nullptr;
    bool dp_pending = false;

    // OFDM
    OfdmState ofdm;
    dabgpu_wideband* wb = nullptr;   // open wideband front end feeding the OFDM stage (dabgpu_wideband_open)

    // dabgpu_submit / dabgpu_wait pipeline
    struct PipeSlot {
        cudaEvent_t h2d_done = nullptr, compute_done = nullptr, d2h_done = nullptr;
        DevBuf d_stage, d_produced;
        DevBuf d_written0;   // frames_written of the ticket's streams before its first OFDM run (dabgpu_wideband_submit)
        DevBuf d_dpout;      // the ticket's packed DAB+ log, then its index (dabgpu_submit_ex / dabgpu_wideband_submit_ex)
        uint64_t ticket = 0;
        bool busy = false;
    } pipe[DABGPU_PIPELINE_DEPTH];
    cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
    uint64_t next_ticket = 1;
    size_t pipe_recent_samples[DABGPU_PIPELINE_DEPTH] = {0, 0};
};

static bool is_pow2(size_t v) { return v && !(v & (v - 1)); }

// the main stream waits for the last channel decode (if it is still running on the channel stream)
static cudaError_t join_dabplus(dabgpu_ctx* ctx) {
    if (!ctx->dp_pending) return cudaSuccess;
    ctx->dp_pending = false;
    return cudaStreamWaitEvent(ctx->stream, ctx->ev_dp, 0);
}
static cudaError_t sync_ctx(dabgpu_ctx* ctx) {
    cudaError_t e = join_dabplus(ctx);
    if (e != cudaSuccess) return e;
    return cudaStreamSynchronize(ctx->stream);
}

static void wb_detach(dabgpu_wideband* w);

// The control kernel divides by the L1 window length and by its stride (signal_l1_nb_samples x nb_decimate): both knobs must
// be positive wherever a configuration enters, at context creation and in dabgpu_ofdm_set_config.
static int validate_ofdm_config(const dabgpu_ofdm_config& c) {
    if (c.signal_l1_nb_samples < 1 || c.signal_l1_nb_decimate < 1)
        return set_error(DABGPU_ERR_INVALID, "signal_l1 window parameters must be >= 1 (nb_samples %d, nb_decimate %d)", c.signal_l1_nb_samples,
                         c.signal_l1_nb_decimate);
    return DABGPU_OK;
}

extern "C" {

const char* dabgpu_version(void) { return DABGPU_VERSION; }
const char* dabgpu_last_error(void) { return g_last_error; }

int dabgpu_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

void dabgpu_config_default(dabgpu_config* cfg, int transmission_mode) {
    memset(cfg, 0, sizeof(*cfg));
    cfg->device = 0;
    cfg->transmission_mode = transmission_mode;
    cfg->max_streams = 1;
    cfg->iq_format = DABGPU_IQ_U8;
    cfg->ring_samples = 0;
    cfg->frame_slots = 0;
    cfg->max_subchannels = 0;
    cfg->cuda_stream = nullptr;
    // OFDM_Demod_Config defaults, ofdm/ofdm_demodulator.h:24-45
    cfg->ofdm.signal_l1_update_beta = 0.95f;
    cfg->ofdm.signal_l1_nb_samples = 100;
    cfg->ofdm.signal_l1_nb_decimate = 5;
    cfg->ofdm.null_thresh_start = 0.35f;
    cfg->ofdm.null_thresh_end = 0.75f;
    cfg->ofdm.fine_freq_update_beta = 0.9f;
    cfg->ofdm.is_coarse_freq_correction = 1;
    cfg->ofdm.max_coarse_freq_correction_norm = 0.5f;
    cfg->ofdm.coarse_freq_slow_beta = 0.1f;
    cfg->ofdm.impulse_peak_threshold_db = 20.0f;
    cfg->ofdm.impulse_peak_distance_probability = 0.15f;
    cfg->flags = 0;
}

int dabgpu_get_params(int transmission_mode, dabgpu_params* out) {
    if (!out) return set_error(DABGPU_ERR_INVALID, "null output");
    return fill_params(transmission_mode, out);
}

static int ensure_scratch(dabgpu_ctx* ctx, uint32_t steps) {
    if (steps <= ctx->scratch_steps) return DABGPU_OK;
    const uint32_t rounded = (steps + 63u) & ~63u;
    const size_t slots = size_t(ctx->vit_blocks) * VIT_WARPS_PER_BLOCK;
    CUDA_TRY(sync_ctx(ctx));
    int rc = ctx->d_scratch.alloc(slots * rounded * sizeof(uint2));
    if (rc) return rc;
    ctx->scratch_steps = rounded;
    return DABGPU_OK;
}

int dabgpu_ctx_create(const dabgpu_config* cfg, dabgpu_ctx** out) {
    if (!cfg || !out) return set_error(DABGPU_ERR_INVALID, "null argument");
    *out = nullptr;
    dabgpu_params P;
    int rc = fill_params(cfg->transmission_mode, &P);
    if (rc) return rc;
    if ((rc = validate_ofdm_config(cfg->ofdm))) return rc;
    if (cfg->max_streams < 1) return set_error(DABGPU_ERR_INVALID, "max_streams must be >= 1");
    if (cfg->iq_format != DABGPU_IQ_U8 && cfg->iq_format != DABGPU_IQ_C32) return set_error(DABGPU_ERR_INVALID, "bad iq_format");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return set_error(DABGPU_ERR_CUDA, "no CUDA device available: libdabgpu has no CPU fallback");
    }
    if (cfg->device < 0 || cfg->device >= ndev) return set_error(DABGPU_ERR_INVALID, "device %d out of range (%d devices)", cfg->device, ndev);
    CUDA_TRY(cudaSetDevice(cfg->device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major < 10) return set_error(DABGPU_ERR_CUDA, "device %s is sm_%d%d; libdabgpu is built for sm_100a only", prop.name, prop.major, prop.minor);

    dabgpu_ctx* ctx = new dabgpu_ctx();
    ctx->cfg = *cfg;
    ctx->P = P;
    ctx->num_sms = prop.multiProcessorCount;
    const int S = cfg->max_streams;
    int min_slots = 8;
    // the time de-interleaver needs 16 CIFs of history plus the frame being written
    while (min_slots * P.nb_cifs < 16 + 2 * P.nb_cifs) min_slots *= 2;
    // default: twice the minimum, so that a consumer may fall several frames behind the OFDM stage before frames are dropped
    ctx->frame_slots = cfg->frame_slots > 0 ? cfg->frame_slots : 2 * min_slots;
    if (!is_pow2(size_t(ctx->frame_slots)) || ctx->frame_slots < min_slots) {
        delete ctx;
        return set_error(DABGPU_ERR_INVALID, "frame_slots must be a power of two >= %d", min_slots);
    }
    ctx->max_subs = cfg->max_subchannels > 0 ? cfg->max_subchannels : 64;
    if (cfg->cuda_stream) {
        ctx->stream = (cudaStream_t)cfg->cuda_stream;
    } else {
        cudaError_t e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) { delete ctx; return set_error(DABGPU_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e)); }
        ctx->own_stream = true;
    }
#define TRY_OR_FREE(expr) do { rc = (expr); if (rc) { dabgpu_ctx_destroy(ctx); return rc; } } while (0)
    TRY_OR_FREE(upload_constant_tables());
    {
        std::vector<uint32_t> w;
        ctx->prbs_words = 2048;   // 8192 bytes >= CIF_OUT_STRIDE
        host_prbs_words(w, ctx->prbs_words);
        TRY_OR_FREE(ctx->d_prbs.alloc(w.size() * 4));
        cudaMemcpy(ctx->d_prbs.p, w.data(), w.size() * 4, cudaMemcpyHostToDevice);
    }
    TRY_OR_FREE(ctx->d_counter.alloc(64));
    // persistent grid: 4 CTAs x 4 warps per SM, each warp with 12.5 KB of decision words in shared memory
    ctx->vit_blocks = ctx->num_sms * 4;
    {
        cudaError_t e = cudaFuncSetAttribute(k_viterbi, cudaFuncAttributeMaxDynamicSharedMemorySize, int(VIT_SMEM_BYTES));
        if (e != cudaSuccess) { rc = set_error(DABGPU_ERR_CUDA, "cudaFuncSetAttribute(k_viterbi): %s", cudaGetErrorString(e)); dabgpu_ctx_destroy(ctx); return rc; }
    }
    {
        cudaError_t e = cudaFuncSetAttribute(k_vit_prep, cudaFuncAttributeMaxDynamicSharedMemorySize, int(VP_SMEM_BYTES));
        if (e != cudaSuccess) { rc = set_error(DABGPU_ERR_CUDA, "cudaFuncSetAttribute(k_vit_prep): %s", cudaGetErrorString(e)); dabgpu_ctx_destroy(ctx); return rc; }
    }
    TRY_OR_FREE(ensure_scratch(ctx, 1600));
    TRY_OR_FREE(ctx->d_vlplan.alloc(sizeof(VlPlan)));
    ctx->vl_mode = (cfg->flags & DABGPU_FLAG_VIT_LANES_ALWAYS) ? 1 : ((cfg->flags & DABGPU_FLAG_VIT_LANES_NEVER) ? 2 : 0);
    if (const char* e = getenv("DABGPU_VIT_LANES")) {   // test hook: run every Viterbi call through one mapping
        if (!strcmp(e, "always")) ctx->vl_mode = 1;
        else if (!strcmp(e, "never")) ctx->vl_mode = 2;
    }
    if (const char* e = getenv("DABGPU_VIT_LANE_CTAS_PER_SM")) { const int k = atoi(e); if (k == 1 || k == 4) ctx->vl_ctas_forced = k; }

    // frame ring + channel decode buffers
    const size_t frame_bits = size_t(P.nb_frame_bits);
    TRY_OR_FREE(ctx->d_frames.alloc(size_t(S) * ctx->frame_slots * frame_bits + 1024));   // + slack: k_vit_prep reads whole 16-byte pieces of a plane / 256-byte units of a FIC group
    TRY_OR_FREE(ctx->d_frames_written.alloc(size_t(S) * 4));
    TRY_OR_FREE(ctx->d_frames_decoded.alloc(size_t(S) * 4));
    TRY_OR_FREE(ctx->d_frames_snapshot.alloc(size_t(S) * 4));
    TRY_OR_FREE(ctx->d_frame_info.alloc(size_t(S) * ctx->frame_slots * sizeof(dabgpu_frame_info)));
    TRY_OR_FREE(ctx->d_subcfg.alloc(size_t(S) * ctx->max_subs * sizeof(SubCfgDev)));
    TRY_OR_FREE(ctx->d_nsubs.alloc(size_t(S) * 4));
    TRY_OR_FREE(ctx->d_cifs_consumed.alloc(size_t(S) * ctx->max_subs * 4));
    TRY_OR_FREE(ctx->d_fic_out.alloc(size_t(S) * P.nb_cifs * FIC_GROUP_BYTES));
    TRY_OR_FREE(ctx->d_fic_crc.alloc(size_t(S) * P.nb_cifs * 4));
    TRY_OR_FREE(ctx->d_msc_out.alloc(size_t(S) * P.nb_cifs * CIF_OUT_STRIDE));
    TRY_OR_FREE(ctx->d_msc_valid.alloc(size_t(S) * P.nb_cifs * ctx->max_subs));
    TRY_OR_FREE(ctx->d_deint.alloc(size_t(S) * P.nb_cifs * P.nb_cif_bits + 1024));   // + slack: k_vit_prep reads whole 256-byte units
    TRY_OR_FREE(ctx->d_status.alloc(size_t(S) * 8));
    TRY_OR_FREE(ctx->d_counters.alloc(CNT_COUNT * 8));
    TRY_OR_FREE(ctx->h_status.alloc(size_t(S) * 8 + 4096));
    cudaMemset(ctx->d_frames.p, 0, ctx->d_frames.bytes);
    cudaMemset(ctx->d_frames_written.p, 0, ctx->d_frames_written.bytes);
    cudaMemset(ctx->d_frames_decoded.p, 0, ctx->d_frames_decoded.bytes);
    cudaMemset(ctx->d_frames_snapshot.p, 0, ctx->d_frames_snapshot.bytes);
    cudaMemset(ctx->d_frame_info.p, 0, ctx->d_frame_info.bytes);
    cudaMemset(ctx->d_subcfg.p, 0, ctx->d_subcfg.bytes);
    cudaMemset(ctx->d_nsubs.p, 0, ctx->d_nsubs.bytes);
    cudaMemset(ctx->d_cifs_consumed.p, 0, ctx->d_cifs_consumed.bytes);
    cudaMemset(ctx->d_fic_out.p, 0, ctx->d_fic_out.bytes);
    cudaMemset(ctx->d_fic_crc.p, 0, ctx->d_fic_crc.bytes);
    cudaMemset(ctx->d_msc_out.p, 0, ctx->d_msc_out.bytes);
    cudaMemset(ctx->d_msc_valid.p, 0, ctx->d_msc_valid.bytes);
    cudaMemset(ctx->d_status.p, 0, ctx->d_status.bytes);
    cudaMemset(ctx->d_counters.p, 0, ctx->d_counters.bytes);
    ctx->subs.resize(size_t(S));
    ctx->h_frames_popped.assign(size_t(S), 0);
    ctx->h_frames_dropped.assign(size_t(S), 0);

    ChanDev& C = ctx->chan;
    C.geom.nb_cifs = uint32_t(P.nb_cifs);
    C.geom.cif_shift = (P.nb_cifs == 4) ? 2u : (P.nb_cifs == 2 ? 1u : 0u);
    C.geom.frame_bits = uint32_t(P.nb_frame_bits);
    C.geom.fic_bits = uint32_t(P.nb_fic_bits);
    C.geom.cif_bits = uint32_t(P.nb_cif_bits);
    C.geom.slot_mask = uint32_t(ctx->frame_slots - 1);
    C.nb_fibs_per_cif = uint32_t(P.nb_fibs_per_cif);
    C.fib_group_bits = uint32_t(P.nb_fib_group_bits);
    // FIC_Decoder only decodes 2304-bit FIB groups (fic_decoder.cpp:66-72): mode III is skipped like the reference
    C.fic_enabled = (P.nb_fib_group_bits == 2304 && !(cfg->flags & DABGPU_FLAG_NO_FIC)) ? 1u : 0u;
    C.max_subs = uint32_t(ctx->max_subs);
    C.jobs_per_stream = uint32_t(P.nb_cifs) * (1u + uint32_t(ctx->max_subs));
    C.frames = ctx->d_frames.as<int8_t>();
    C.stream_frames_stride = size_t(ctx->frame_slots) * frame_bits;
    C.frames_written = ctx->d_frames_snapshot.as<uint32_t>();
    C.frames_decoded = ctx->d_frames_decoded.as<uint32_t>();
    C.subcfg = ctx->d_subcfg.as<SubCfgDev>();
    C.n_subs = ctx->d_nsubs.as<uint32_t>();
    C.cifs_consumed = ctx->d_cifs_consumed.as<uint32_t>();
    C.fic_out = ctx->d_fic_out.as<uint8_t>();
    C.fic_crc = ctx->d_fic_crc.as<uint8_t>();
    C.msc_out = ctx->d_msc_out.as<uint8_t>();
    C.msc_valid = ctx->d_msc_valid.as<uint8_t>();
    C.deint = ctx->d_deint.as<int8_t>();
    C.status = ctx->d_status.as<int32_t>();
    C.counters = ctx->d_counters.as<unsigned long long>();

    TRY_OR_FREE(dabplus_init(ctx->dabplus, S, ctx->max_subs, P.nb_cifs));
    if (getenv("DABGPU_CHAN_INLINE") == nullptr) {   // A/B switch: keep the channel decode on the main stream
        int prio_lo = 0, prio_hi = 0;
        cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
        // the channel stream gets the higher priority: its CTAs are placed as soon as the demodulator's retire, instead of
        // after the whole queued wave (2.97 -> 2.75 ms per 1024-stream step); DABGPU_CHAN_PRIO_OFF is the A/B switch
        const int dp_prio = getenv("DABGPU_CHAN_PRIO_OFF") ? prio_lo : prio_hi;
        if (cudaStreamCreateWithPriority(&ctx->s_dp, cudaStreamNonBlocking, dp_prio) != cudaSuccess || cudaEventCreateWithFlags(&ctx->ev_dp, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&ctx->ev_dp_fork, cudaEventDisableTiming) != cudaSuccess) {
            rc = set_error(DABGPU_ERR_CUDA, "DAB+ stream / event creation failed");
            dabgpu_ctx_destroy(ctx);
            return rc;
        }
    }
    {
        // Decoding frame t gathers CIFs newest-15 .. newest, i.e. the frames t-hist .. t; the newest written frame w-1 shares a
        // slot with frame w-1-slots, so the history is intact while w - t <= slots - hist.  When the channel decode runs on its
        // own stream the next OFDM stage may write up to two more frames meanwhile (dabgpu_ofdm_* joins first when a call can
        // emit more than that), hence two slots of margin.
        const int hist = (15 + P.nb_cifs - 1) / P.nb_cifs;
        const int lag = ctx->frame_slots - hist - (ctx->s_dp ? 2 : 0);
        C.max_lag = uint32_t(lag < 1 ? 1 : lag);
    }
    ctx->ofdm.prof = &ctx->prof;
    TRY_OR_FREE(ofdm_init(ctx->ofdm, ctx->cfg, P, ctx->frame_slots, ctx->d_frames.as<int8_t>(), ctx->d_frames_written.as<uint32_t>(),
                          ctx->d_frame_info.as<dabgpu_frame_info>(), ctx->d_counters.as<unsigned long long>()));
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { dabgpu_ctx_destroy(ctx); return set_error(DABGPU_ERR_CUDA, "context initialisation: %s", cudaGetErrorString(e)); }
    *out = ctx;
    return DABGPU_OK;
}

void dabgpu_ctx_destroy(dabgpu_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->cfg.device);
    if (ctx->stream) sync_ctx(ctx);
    ctx->prof.destroy();
    for (auto& sl : ctx->pipe) {
        if (sl.h2d_done) cudaEventDestroy(sl.h2d_done);
        if (sl.compute_done) cudaEventDestroy(sl.compute_done);
        if (sl.d2h_done) cudaEventDestroy(sl.d2h_done);
        sl.d_stage.release();
        sl.d_produced.release();
        sl.d_written0.release();
        sl.d_dpout.release();
    }
    if (ctx->s_dp) { cudaStreamSynchronize(ctx->s_dp); cudaStreamDestroy(ctx->s_dp); }
    if (ctx->ev_dp) cudaEventDestroy(ctx->ev_dp);
    if (ctx->ev_dp_fork) cudaEventDestroy(ctx->ev_dp_fork);
    if (ctx->s_h2d) { cudaStreamSynchronize(ctx->s_h2d); cudaStreamDestroy(ctx->s_h2d); }
    if (ctx->wb) wb_detach(ctx->wb);
    if (ctx->s_d2h) { cudaStreamSynchronize(ctx->s_d2h); cudaStreamDestroy(ctx->s_d2h); }
    ofdm_destroy(ctx->ofdm);
    dabplus_destroy(ctx->dabplus);
    packet_destroy(ctx->packet);
    DevBuf* bufs[] = {&ctx->d_vlplan, &ctx->d_vllist, &ctx->d_vlsym, &ctx->d_vlscratch, &ctx->d_prbs, &ctx->d_counter, &ctx->d_scratch, &ctx->d_jobs, &ctx->d_vsoft, &ctx->d_vout, &ctx->d_verr,
                      &ctx->d_frames, &ctx->d_frames_written, &ctx->d_frames_decoded, &ctx->d_frames_snapshot, &ctx->d_pushstage, &ctx->d_popstage, &ctx->d_frame_info, &ctx->d_subcfg, &ctx->d_nsubs,
                      &ctx->d_cifs_consumed, &ctx->d_fic_out, &ctx->d_fic_crc, &ctx->d_msc_out, &ctx->d_msc_valid, &ctx->d_deint, &ctx->d_status,
                      &ctx->d_counters};
    for (DevBuf* b : bufs) b->release();
    ctx->h_status.release();
    ctx->h_stage.release();
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

// Pinned host memory for dabgpu_submit / dabgpu_ofdm_process buffers.  write_combined: for buffers the CPU only writes (the IQ
// the host feeds in): uncached on the CPU side, so the copy engine's reads do not snoop the CPU caches.
int dabgpu_host_alloc(void** out, size_t bytes, int write_combined) {
    if (!out) return set_error(DABGPU_ERR_INVALID, "null output");
    *out = nullptr;
    const cudaError_t e = cudaHostAlloc(out, bytes, write_combined ? cudaHostAllocWriteCombined : cudaHostAllocDefault);
    if (e != cudaSuccess) { cudaGetLastError(); return set_error(DABGPU_ERR_NOMEM, "cudaHostAlloc(%zu) failed: %s", bytes, cudaGetErrorString(e)); }
    return DABGPU_OK;
}
void dabgpu_host_free(void* p) { if (p) cudaFreeHost(p); }

int dabgpu_sync(dabgpu_ctx* ctx) {
    if (!ctx) return set_error(DABGPU_ERR_INVALID, "null context");
    CUDA_TRY(sync_ctx(ctx));
    return DABGPU_OK;
}

void* dabgpu_cuda_stream(dabgpu_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
uint64_t dabgpu_launch_count(const dabgpu_ctx* ctx) { return ctx ? ctx->launches + ctx->ofdm.launches : 0; }

int dabgpu_profile_enable(dabgpu_ctx* ctx, int on) {
    if (!ctx) return set_error(DABGPU_ERR_INVALID, "null context");
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    ctx->prof.reset();
    ctx->prof.on = on != 0;
    return DABGPU_OK;
}

int dabgpu_profile_read(dabgpu_ctx* ctx, dabgpu_profile* out) {
    if (!ctx || !out) return set_error(DABGPU_ERR_INVALID, "null argument");
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(sync_ctx(ctx));
    ctx->prof.collect();
    for (int i = 0; i < PROF_CLASSES; i++) { out->ms[i] = ctx->prof.ms[i]; out->launches[i] = ctx->prof.n[i]; }
    return DABGPU_OK;
}

// ---------------------------------------------------------------------------------------------
// Viterbi
// ---------------------------------------------------------------------------------------------
// Host-side upper bound of what a call can contain (per length class), used to size the buffers of the lane path.
struct VlBound {
    uint32_t count[VL_BUCKETS];
    uint32_t max_steps = 0;
    bool oversize = false;
    VlBound() { memset(count, 0, sizeof(count)); }
    void add(uint32_t steps, uint32_t n = 1) {
        if (steps == 0 || n == 0) return;
        if (steps >= VL_MAX_STEPS) { oversize = true; return; }
        count[vl_bucket(steps)] += n;
        if (steps > max_steps) max_steps = steps;
    }
    void totals(uint32_t* rows, uint32_t* groups, uint32_t* active) const {
        uint64_t r = 0, g = 0, a = 0;
        for (uint32_t b = 0; b < VL_BUCKETS; b++) {
            const uint64_t gb = (count[b] + 31u) >> 5;
            g += gb; r += gb * vl_bucket_rows(b); a += count[b];
        }
        *rows = r > 0xFFFFFFFFull ? 0xFFFFFFFFu : uint32_t(r); *groups = uint32_t(g); *active = uint32_t(a);
    }
};

#define VIT_ORDER_MIN_JOBS 1024u   // calls with at least this many trellises that stay on k_viterbi are decoded longest first
#ifndef VL_TB_WIDE
#define VL_TB_WIDE 10u   // traceback rows per batch of the 128-register lane kernel (two batches in flight); 15 / 20 / 25 rows hide more of
                         // the decision loads' latency but spill in the forward loop: 1.26 / 1.25 / 1.39 ms against 1.13
#endif
static int launch_viterbi(dabgpu_ctx* ctx, const VitJobDev* d_jobs, int n_jobs, const VlBound* bound, bool precounted = false) {
    CUDA_TRY(cudaMemsetAsync(ctx->d_counter.p, 0, 4, ctx->stream));
    VlPlan* plan = nullptr;
    VlPlan* order_plan = nullptr;      // plan used only to order k_viterbi's queue
    uint32_t rows = 0, groups = 0, active = 0;
    bool lanes_wide = false;
    if (bound && !bound->oversize && ctx->vl_mode != 2) {
        bound->totals(&rows, &groups, &active);
        // rows * 128 B of symbols: keep the lane path for calls whose symbol matrix stays below 16 GiB
        if (active > 0 && (ctx->vl_mode == 1 || active >= ctx->vl_min_jobs) && uint64_t(rows) * 128u <= (16ull << 30)) {
            int rc;
            const uint32_t need_rows = bound->max_steps + 64u;
            lanes_wide = ctx->vl_ctas_forced == 4 || (ctx->vl_ctas_forced == 0 && groups > uint32_t(ctx->num_sms) * VL_WARPS_PER_BLOCK * 2u);
            const uint32_t need_slots = uint32_t(ctx->num_sms) * VL_WARPS_PER_BLOCK * (lanes_wide ? 4u : 1u);
            if (need_rows > ctx->vl_scratch_rows || need_slots > ctx->vl_scratch_slots || !ctx->d_vlscratch.p) {
                CUDA_TRY(sync_ctx(ctx));
                const uint32_t r = std::max((need_rows + 255u) & ~255u, ctx->vl_scratch_rows);
                const uint32_t sl = std::max(need_slots, ctx->vl_scratch_slots);
                if ((rc = ctx->d_vlscratch.alloc(size_t(sl) * r * 32u * sizeof(uint2)))) return rc;
                ctx->vl_scratch_rows = r;
                ctx->vl_scratch_slots = sl;
            }
            if (ctx->d_vllist.bytes < size_t(n_jobs) * 4 || ctx->d_vlsym.bytes < size_t(rows) * 128u) CUDA_TRY(sync_ctx(ctx));
            if ((rc = ctx->d_vllist.alloc(size_t(n_jobs) * 4))) return rc;
            if ((rc = ctx->d_vlsym.alloc(size_t(rows) * 128u))) return rc;
            plan = ctx->d_vlplan.as<VlPlan>();
        } else if (active >= VIT_ORDER_MIN_JOBS) {
            // too few trellises for the lane kernel, enough for the order to matter: k_viterbi pulls them longest first (below)
            int rc;
            if (ctx->d_vllist.bytes < size_t(n_jobs) * 4) CUDA_TRY(sync_ctx(ctx));
            if ((rc = ctx->d_vllist.alloc(size_t(n_jobs) * 4))) return rc;
            order_plan = ctx->d_vlplan.as<VlPlan>();
        }
    }
    if (order_plan) {
        // A call that mixes short and long trellises (UEP row 63 is 9 222 steps, a FIB group 774) leaves its longest jobs to the end
        // of k_viterbi's queue in job order, and the call then waits for a few warps walking the longest trellises alone.  The lane
        // path's histogram and scatter give the job list by length class, longest first (1.11 instead of 1.35 ms for 256 streams of
        // UEP rows 0 / 14 / 37 / 63: what remains is one warp's walk over 9 222 steps).  Scheduling only: every trellis is decoded by the same code.
        ctx->prof.begin(PROF_CHAN_MISC, ctx->stream);
        const int tb = 256, nb = (n_jobs + tb - 1) / tb;
        if (!precounted) {
            CUDA_TRY(cudaMemsetAsync(order_plan, 0, sizeof(VlPlan), ctx->stream));
            k_vit_count<<<nb, tb, 0, ctx->stream>>>(d_jobs, n_jobs, order_plan);
        }
        k_vit_plan<<<1, 32, 0, ctx->stream>>>(order_plan, 2 /* never the lane kernel */, 0u, 0u, 0u);
        k_vit_scatter<<<nb, tb, 0, ctx->stream>>>(d_jobs, n_jobs, order_plan, ctx->d_vllist.as<uint32_t>());
        ctx->prof.end(ctx->stream);
        ctx->launches += precounted ? 2 : 3;
    }
    if (plan) {
        static const VlConst kc = {0xFFFFFFFFu, 2u, 4u, 16u, 256u, 0x10000u};
        // planning + time de-interleave / de-puncture pass are accounted as "chan_misc", the decoders as "viterbi"
        ctx->prof.begin(PROF_CHAN_MISC, ctx->stream);
        const int tb = 256, nb = (n_jobs + tb - 1) / tb;
        if (!precounted) {   // dabgpu_chan_decode takes the histogram while it builds the jobs
            CUDA_TRY(cudaMemsetAsync(plan, 0, sizeof(VlPlan), ctx->stream));
            k_vit_count<<<nb, tb, 0, ctx->stream>>>(d_jobs, n_jobs, plan);
        }
        k_vit_plan<<<1, 32, 0, ctx->stream>>>(plan, ctx->vl_mode, ctx->vl_min_jobs, rows, groups);
        k_vit_scatter<<<nb, tb, 0, ctx->stream>>>(d_jobs, n_jobs, plan, ctx->d_vllist.as<uint32_t>());
        // enough warps to fill the GPU: a group's steps are split over up to eight warps
        uint32_t split = 1u;
        while (split < 8u && groups * split * 2u <= uint32_t(ctx->num_sms) * 48u) split *= 2u;
        if (groups * split < uint32_t(ctx->num_sms) * 48u && split < 8u) split *= 2u;
        if (const char* e = getenv("DABGPU_PREP_SPLIT")) { const int v = atoi(e); if (v >= 1 && v <= 16) split = uint32_t(v); }   // tuning knob
        k_vit_prep<<<(groups * split + VP_WARPS - 1u) / VP_WARPS, VP_WARPS * 32, VP_SMEM_BYTES, ctx->stream>>>(d_jobs, plan, ctx->d_vllist.as<uint32_t>(),
                                                                                                       ctx->d_vlsym.as<uint32_t>(), ctx->chan.geom, split);
        ctx->prof.end(ctx->stream);
        ctx->prof.begin(PROF_VITERBI, ctx->stream);
        if (!lanes_wide) {
            k_viterbi_lanes<40u, 1><<<ctx->num_sms, VL_WARPS_PER_BLOCK * 32, 0, ctx->stream>>>(d_jobs, plan, ctx->d_vllist.as<uint32_t>(), ctx->d_vlsym.as<uint32_t>(),
                                                                                            ctx->d_vlscratch.as<uint2>(), ctx->vl_scratch_rows,
                                                                                            ctx->d_prbs.as<uint32_t>(), kc);
        } else {
            // Three CTAs per SM, not the four that fit: 1.12 against 1.21 ms per 1024-stream call on its own (three warps per
            // sub-partition each run faster, the short second wave costs less than that gains).  In a receiver loop the OFDM stage
            // of the next step runs on the other stream meanwhile; the demodulator is then capped at three CTAs per SM as well, so
            // that one of its CTAs always fits beside the lane kernel's three: 2.28 ms per 1024-stream step against 2.33 for four +
            // four, 2.45 for two + two and 2.49 run one after the other (profiles/r2_coresidency_c.txt).
            int per_sm = 3;
            // a call with slightly more groups than warps would run a second, nearly empty wave of whole trellises: one CTA more
            {
                const uint32_t slots = uint32_t(ctx->num_sms) * VL_WARPS_PER_BLOCK * uint32_t(per_sm);
                if (groups > slots && groups * 4u < slots * 5u) per_sm++;
            }
            if (const char* e = getenv("DABGPU_LANES_CTAS")) { const int v = atoi(e); if (v >= 1 && v <= 4) per_sm = v; }   // tuning knob
            k_viterbi_lanes<VL_TB_WIDE, 4><<<ctx->num_sms * per_sm, VL_WARPS_PER_BLOCK * 32, 0, ctx->stream>>>(d_jobs, plan, ctx->d_vllist.as<uint32_t>(), ctx->d_vlsym.as<uint32_t>(),
                                                                                                ctx->d_vlscratch.as<uint2>(), ctx->vl_scratch_rows,
                                                                                                ctx->d_prbs.as<uint32_t>(), kc);
        }
        ctx->launches += precounted ? 4 : 5;
    } else {
        ctx->prof.begin(PROF_VITERBI, ctx->stream);
    }
    // the warp-per-trellis kernel takes the call when the plan says so (few trellises, or no plan at all)
    k_viterbi<<<ctx->vit_blocks, VIT_WARPS_PER_BLOCK * 32, VIT_SMEM_BYTES, ctx->stream>>>(d_jobs, n_jobs, ctx->d_counter.as<int>(), ctx->d_scratch.as<uint2>(),
                                                                                       ctx->scratch_steps, ctx->d_prbs.as<uint32_t>(), ctx->chan.geom,
                                                                                       reinterpret_cast<const uint32_t*>(plan ? plan : order_plan),
                                                                                       (plan || order_plan) ? ctx->d_vllist.as<uint32_t>() : nullptr);
    ctx->prof.end(ctx->stream);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return DABGPU_OK;
}

int dabgpu_viterbi_decode(dabgpu_ctx* ctx, const dabgpu_viterbi_job* jobs, int n_jobs, const int8_t* soft_host, size_t soft_bytes,
                          uint8_t* out_host, size_t out_bytes, uint64_t* path_error_host) {
    if (!ctx || !jobs || !soft_host || !out_host) return set_error(DABGPU_ERR_INVALID, "null argument");
    if (n_jobs <= 0) return DABGPU_OK;
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(join_dabplus(ctx));   // shares the job, plan and scratch buffers with a channel decode that may still be running
    int rc;
    if ((rc = ctx->d_vsoft.alloc(soft_bytes + 1024))) return rc;   // k_vit_prep reads whole 256-byte units
    if ((rc = ctx->d_vout.alloc(out_bytes + 16))) return rc;
    if ((rc = ctx->d_verr.alloc(size_t(n_jobs) * 8))) return rc;
    if ((rc = ctx->d_jobs.alloc(size_t(n_jobs) * sizeof(VitJobDev)))) return rc;
    std::vector<VitJobDev> hj(static_cast<size_t>(n_jobs));
    uint32_t max_steps = 0;
    VlBound vb;
    for (int i = 0; i < n_jobs; i++) {
        const dabgpu_viterbi_job& j = jobs[i];
        VitJobDev& J = hj[size_t(i)];
        memset(&J, 0, sizeof(J));
        if (j.n_seg < 1 || j.n_seg > DABGPU_MAX_SEGMENTS) return set_error(DABGPU_ERR_INVALID, "job %d: n_seg %u out of range", i, j.n_seg);
        uint32_t steps = 0, in_base = 0;
        for (uint32_t k = 0; k < DABGPU_MAX_SEGMENTS; k++) {
            if (k < j.n_seg) {
                if (j.seg_pi[k] > 24) return set_error(DABGPU_ERR_INVALID, "job %d: puncture code %u out of range", i, j.seg_pi[k]);
                if (j.seg_bits[k] % 4 != 0) return set_error(DABGPU_ERR_INVALID, "job %d: segment bits must be a multiple of the code rate", i);
                J.seg_pi[k] = j.seg_pi[k];
                J.seg_in_base[k] = in_base;
                int c[8];
                host_pi_counts(j.seg_pi[k], c);
                const uint32_t groups = j.seg_bits[k] / 4;
                uint32_t per8 = 0;
                for (int g = 0; g < 8; g++) per8 += uint32_t(c[g]);
                in_base += (groups / 8) * per8;
                for (uint32_t g = 0; g < groups % 8; g++) in_base += uint32_t(c[g]);
                steps += groups;
            }
            J.seg_step_end[k] = steps;
        }
        if (in_base > j.n_soft) return set_error(DABGPU_ERR_INVALID, "job %d: needs %u punctured symbols, only %u given", i, in_base, j.n_soft);
        if (j.soft_offset > soft_bytes || j.n_soft > soft_bytes - j.soft_offset) return set_error(DABGPU_ERR_INVALID, "job %d: soft range exceeds buffer", i);
        if (size_t(j.n_out_bytes) * 8 + 6 > steps) return set_error(DABGPU_ERR_INVALID, "job %d: chainback of %u bytes exceeds %u decoded steps", i, j.n_out_bytes, steps);
        if (j.out_offset > out_bytes || j.n_out_bytes > out_bytes - j.out_offset) return set_error(DABGPU_ERR_INVALID, "job %d: output range exceeds buffer", i);
        if (j.descramble && (j.n_out_bytes + 3) / 4 > ctx->prbs_words) return set_error(DABGPU_ERR_INVALID, "job %d: too long for the PRBS table", i);
        J.n_seg = j.n_seg;
        J.total_steps = steps;
        J.n_out_bytes = j.n_out_bytes;
        J.flags = j.descramble ? VJ_DESCRAMBLE : 0u;
        J.src = ctx->d_vsoft.as<int8_t>() + j.soft_offset;
        J.out = ctx->d_vout.as<uint8_t>() + j.out_offset;
        J.path_error = ctx->d_verr.as<unsigned long long>() + i;
        if (steps > max_steps) max_steps = steps;
        vb.add(steps);
    }
    if ((rc = ensure_scratch(ctx, max_steps))) return rc;
    CUDA_TRY(cudaMemcpyAsync(ctx->d_vsoft.p, soft_host, soft_bytes, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(ctx->d_jobs.p, hj.data(), hj.size() * sizeof(VitJobDev), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaMemsetAsync(ctx->d_vout.p, 0, out_bytes, ctx->stream));
    if ((rc = launch_viterbi(ctx, ctx->d_jobs.as<VitJobDev>(), n_jobs, &vb))) return rc;
    CUDA_TRY(cudaMemcpyAsync(out_host, ctx->d_vout.p, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (path_error_host) CUDA_TRY(cudaMemcpyAsync(path_error_host, ctx->d_verr.p, size_t(n_jobs) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(sync_ctx(ctx));
    return DABGPU_OK;
}

// ---------------------------------------------------------------------------------------------
// Channel decode of frames
// ---------------------------------------------------------------------------------------------
static int check_stream_range(dabgpu_ctx* ctx, int first, int n) {
    if (!ctx) return set_error(DABGPU_ERR_INVALID, "null context");
    if (first < 0 || n < 0 || first + n > ctx->cfg.max_streams) return set_error(DABGPU_ERR_INVALID, "stream range [%d,%d) outside [0,%d)", first, first + n, ctx->cfg.max_streams);
    return DABGPU_OK;
}

// Validates one sub-channel description and builds its host / device records (out_offset is assigned by the caller).
static int build_sub(dabgpu_ctx* ctx, const dabgpu_subchannel_ex& ex, int index, SubHost* h, SubCfgDev* d) {
    const dabgpu_subchannel& sc = ex.sc;
    h->sc = sc;
    h->payload = ex.payload;
    h->active = true;
    if (ex.payload < DABGPU_PAYLOAD_STREAM || ex.payload > DABGPU_PAYLOAD_PACKET_FEC)
        return set_error(DABGPU_ERR_INVALID, "sub-channel %d: unknown payload kind %d", index, ex.payload);
    if (h->is_packet() && sc.is_dabplus) return set_error(DABGPU_ERR_INVALID, "sub-channel %d: a packet-mode sub-channel cannot be DAB+", index);
    if ((ex.payload == DABGPU_PAYLOAD_DABPLUS) != (sc.is_dabplus != 0))
        return set_error(DABGPU_ERR_INVALID, "sub-channel %d: payload %d disagrees with is_dabplus %d", index, ex.payload, sc.is_dabplus);
    if (sc.start_address < 0 || sc.length <= 0 || (sc.start_address + sc.length) * 64 > ctx->P.nb_cif_bits)
        return set_error(DABGPU_ERR_INVALID, "Subchannel bits %d:%d overflows MSC channel with %d bits", sc.start_address * 64,
                         (sc.start_address + sc.length) * 64, ctx->P.nb_cif_bits);
    int rc;
    if ((rc = make_schedule(sc, &h->sched))) return rc;
    const int steps = h->sched.total_steps();
    if (h->sched.punctured_bits() > sc.length * 64)
        return set_error(DABGPU_ERR_INVALID, "sub-channel %d: protection profile needs %d soft bits, sub-channel has %d", index, h->sched.punctured_bits(), sc.length * 64);
    h->n_out_bytes = uint32_t((steps - 6) / 8);
    h->out_offset = 0;
    memset(d, 0, sizeof(*d));
    d->start_bit = uint32_t(sc.start_address * 64);
    d->nb_bits = uint32_t(sc.length * 64);
    uint32_t st = 0, inb = 0;
    for (int k = 0; k < DABGPU_MAX_SEGMENTS; k++) {
        if (k < h->sched.n_seg) {
            d->seg_pi[k] = uint8_t(h->sched.pi[k]);
            d->seg_in_base[k] = inb;
            int c[8];
            host_pi_counts(h->sched.pi[k], c);
            const uint32_t groups = uint32_t(h->sched.bits[k] / 4);
            uint32_t per8 = 0;
            for (int g = 0; g < 8; g++) per8 += uint32_t(c[g]);
            inb += (groups / 8) * per8;
            for (uint32_t g = 0; g < groups % 8; g++) inb += uint32_t(c[g]);
            st += groups;
        }
        d->seg_step_end[k] = st;
    }
    d->n_seg = uint32_t(h->sched.n_seg);
    d->total_steps = uint32_t(steps);
    d->n_out_bytes = h->n_out_bytes;
    d->is_dabplus = sc.is_dabplus ? 1u : 0u;
    d->payload = uint32_t(ex.payload);
    return DABGPU_OK;
}

static dabgpu_subchannel_ex sub_ex(const dabgpu_subchannel& sc) {
    dabgpu_subchannel_ex ex;
    ex.sc = sc;
    ex.payload = sc.is_dabplus ? DABGPU_PAYLOAD_DABPLUS : DABGPU_PAYLOAD_STREAM;
    return ex;
}

static bool same_subchannel(const SubHost& x, const SubHost& y) {
    const dabgpu_subchannel &a = x.sc, &b = y.sc;
    if (x.payload != y.payload) return false;
    if (a.start_address != b.start_address || a.length != b.length || (a.is_uep != 0) != (b.is_uep != 0) || (a.is_dabplus != 0) != (b.is_dabplus != 0)) return false;
    return a.is_uep ? (a.uep_prot_index == b.uep_prot_index) : (a.eep_prot_level == b.eep_prot_level && (a.eep_type_b != 0) == (b.eep_type_b != 0));
}

// Writes entry `index` of a stream's sub-channel table to the device; `fresh` also empties its time de-interleaver and DAB+
// superframe state (a new MSC_Decoder + AAC_Frame_Processor), otherwise the running state is left alone.
static int upload_sub(dabgpu_ctx* ctx, int stream, int index, const SubCfgDev& d, bool fresh) {
    const size_t idx = size_t(stream) * ctx->max_subs + size_t(index);
    CUDA_TRY(cudaMemcpy(ctx->d_subcfg.as<SubCfgDev>() + idx, &d, sizeof(SubCfgDev), cudaMemcpyHostToDevice));
    if (fresh) {
        CUDA_TRY(cudaMemset(ctx->d_cifs_consumed.as<uint32_t>() + idx, 0, 4));
        CUDA_TRY(cudaMemset(ctx->dabplus.dev.st + idx, 0, sizeof(DabPlusSubState)));
        CUDA_TRY(cudaMemset(ctx->dabplus.dev.n_events + idx, 0, 4));
    }
    return DABGPU_OK;
}

static int upload_nsubs(dabgpu_ctx* ctx, int stream, size_t n) {
    const uint32_t ns = uint32_t(n);
    CUDA_TRY(cudaMemcpy(ctx->d_nsubs.as<uint32_t>() + stream, &ns, 4, cudaMemcpyHostToDevice));
    ctx->cfg_epoch++;
    return DABGPU_OK;
}

// BasicRadio keeps the decoders it already has when the database grows (basic_radio.cpp:98-131): entries of the new table that
// are identical to the entry at the same index of the old one -- same description, same place in the output arena -- keep their
// time de-interleaver and superframe state; every other entry starts empty like a new MSC_Decoder.
int dabgpu_msc_configure(dabgpu_ctx* ctx, int stream, const dabgpu_subchannel* subs, int n_subs) {
    int rc = check_stream_range(ctx, stream, 1);
    if (rc) return rc;
    if (n_subs < 0 || n_subs > ctx->max_subs) return set_error(DABGPU_ERR_INVALID, "n_subs %d exceeds max_subchannels %d", n_subs, ctx->max_subs);
    if (n_subs > 0 && !subs) return set_error(DABGPU_ERR_INVALID, "null sub-channel table");
    std::vector<dabgpu_subchannel_ex> ex(static_cast<size_t>(n_subs));
    for (int i = 0; i < n_subs; i++) ex[size_t(i)] = sub_ex(subs[i]);
    return dabgpu_msc_configure_ex(ctx, stream, ex.data(), n_subs);
}

// A packet entry's region: kept from the old entry it continues, else a fresh one.  Call with the context synchronised.
static int pkt_attach(dabgpu_ctx* ctx, SubHost& h, const SubHost* kept) {
    if (!h.is_packet()) return DABGPU_OK;
    if (kept) { h.pkt_region = kept->pkt_region; h.pkt_cap = kept->pkt_cap; return DABGPU_OK; }
    h.pkt_cap = pkt_item_bound(uint32_t(ctx->P.nb_cifs), h.n_out_bytes);
    uint64_t region = 0;
    int rc = pkt_region_acquire(ctx->packet, h.pkt_cap, &region);
    if (rc) return rc;
    h.pkt_region = int64_t(region);
    return DABGPU_OK;
}
static void pkt_detach(dabgpu_ctx* ctx, SubHost& h) {
    if (h.pkt_region >= 0) pkt_region_release(ctx->packet, h.pkt_cap, uint64_t(h.pkt_region));
    h.pkt_region = -1;
}

int dabgpu_msc_configure_ex(dabgpu_ctx* ctx, int stream, const dabgpu_subchannel_ex* subs, int n_subs) {
    int rc = check_stream_range(ctx, stream, 1);
    if (rc) return rc;
    if (n_subs < 0 || n_subs > ctx->max_subs) return set_error(DABGPU_ERR_INVALID, "n_subs %d exceeds max_subchannels %d", n_subs, ctx->max_subs);
    if (n_subs > 0 && !subs) return set_error(DABGPU_ERR_INVALID, "null sub-channel table");
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    std::vector<SubHost> hs(static_cast<size_t>(n_subs));
    std::vector<SubCfgDev> dev(static_cast<size_t>(n_subs));
    uint32_t out_off = 0, max_steps = 0;
    for (int i = 0; i < n_subs; i++) {
        if ((rc = build_sub(ctx, subs[i], i, &hs[size_t(i)], &dev[size_t(i)]))) return rc;
        hs[size_t(i)].out_offset = dev[size_t(i)].out_offset = out_off;
        out_off += (hs[size_t(i)].n_out_bytes + 15u) & ~15u;
        if (out_off > CIF_OUT_STRIDE) return set_error(DABGPU_ERR_OVERFLOW, "decoded bytes per CIF exceed %u", CIF_OUT_STRIDE);
        max_steps = std::max(max_steps, dev[size_t(i)].total_steps);
    }
    if ((rc = ensure_scratch(ctx, max_steps))) return rc;
    CUDA_TRY(sync_ctx(ctx));
    std::vector<SubHost>& old = ctx->subs[size_t(stream)];
    std::vector<bool> kept(std::max(old.size(), size_t(n_subs)), false);
    for (int i = 0; i < n_subs; i++)
        kept[size_t(i)] = size_t(i) < old.size() && old[size_t(i)].active && old[size_t(i)].out_offset == hs[size_t(i)].out_offset &&
                          same_subchannel(old[size_t(i)], hs[size_t(i)]);
    // packet regions of the new table first: when the pool cannot grow, the regions taken so far go back and the context keeps
    // the old table, its regions and its item list untouched
    for (int i = 0; i < n_subs; i++)
        if ((rc = pkt_attach(ctx, hs[size_t(i)], kept[size_t(i)] ? &old[size_t(i)] : nullptr))) {
            for (int j = 0; j < i; j++)
                if (!kept[size_t(j)]) pkt_detach(ctx, hs[size_t(j)]);
            return rc;
        }
    for (int i = 0; i < n_subs; i++)
        if ((rc = upload_sub(ctx, stream, i, dev[size_t(i)], !kept[size_t(i)]))) return rc;
    for (size_t i = 0; i < old.size(); i++)
        if (!kept[i]) pkt_detach(ctx, old[i]);
    ctx->subs[size_t(stream)] = hs;
    return upload_nsubs(ctx, stream, hs.size());
}

// Attaches a decoder to one more sub-channel of a stream without touching the running ones (BasicRadio::UpdateAfterProcessing,
// basic_radio.cpp:98-131).  *sub_index_out = its index for dabgpu_chan_get_msc / _get_dabplus_events / dabgpu_msc_get_layout.
int dabgpu_msc_add_subchannel(dabgpu_ctx* ctx, int stream, const dabgpu_subchannel* sub, int* sub_index_out) {
    if (!sub) return set_error(DABGPU_ERR_INVALID, "null sub-channel");
    const dabgpu_subchannel_ex ex = sub_ex(*sub);
    return dabgpu_msc_add_subchannel_ex(ctx, stream, &ex, sub_index_out);
}

int dabgpu_msc_add_subchannel_ex(dabgpu_ctx* ctx, int stream, const dabgpu_subchannel_ex* sub, int* sub_index_out) {
    int rc = check_stream_range(ctx, stream, 1);
    if (rc) return rc;
    if (!sub) return set_error(DABGPU_ERR_INVALID, "null sub-channel");
    std::vector<SubHost>& hs = ctx->subs[size_t(stream)];
    if (int(hs.size()) >= ctx->max_subs) return set_error(DABGPU_ERR_OVERFLOW, "sub-channel table of stream %d is full (%d entries)", stream, ctx->max_subs);
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    SubHost h;
    SubCfgDev d;
    if ((rc = build_sub(ctx, *sub, int(hs.size()), &h, &d))) return rc;
    uint32_t out_off = 0;
    for (const SubHost& o : hs) out_off = std::max(out_off, o.out_offset + ((o.n_out_bytes + 15u) & ~15u));
    if (out_off + h.n_out_bytes > CIF_OUT_STRIDE) return set_error(DABGPU_ERR_OVERFLOW, "decoded bytes per CIF exceed %u", CIF_OUT_STRIDE);
    h.out_offset = d.out_offset = out_off;
    if ((rc = ensure_scratch(ctx, d.total_steps))) return rc;
    CUDA_TRY(sync_ctx(ctx));
    if ((rc = pkt_attach(ctx, h, nullptr))) return rc;
    if ((rc = upload_sub(ctx, stream, int(hs.size()), d, true))) {
        pkt_detach(ctx, h);
        return rc;
    }
    hs.push_back(h);
    if (sub_index_out) *sub_index_out = int(hs.size()) - 1;
    return upload_nsubs(ctx, stream, hs.size());
}

// Detaches the decoder of one sub-channel; the indices of the others do not change (the slot stays reserved until a
// dabgpu_msc_configure).  The reference never removes a decoder; this exists for hosts that retune a service.
int dabgpu_msc_remove_subchannel(dabgpu_ctx* ctx, int stream, int sub_index) {
    int rc = check_stream_range(ctx, stream, 1);
    if (rc) return rc;
    std::vector<SubHost>& hs = ctx->subs[size_t(stream)];
    if (sub_index < 0 || size_t(sub_index) >= hs.size() || !hs[size_t(sub_index)].active) return set_error(DABGPU_ERR_INVALID, "sub-channel index %d not configured", sub_index);
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(sync_ctx(ctx));
    SubCfgDev d;
    memset(&d, 0, sizeof(d));   // total_steps = 0: k_chan_build_jobs emits no job and marks every CIF invalid
    d.out_offset = hs[size_t(sub_index)].out_offset;
    if ((rc = upload_sub(ctx, stream, sub_index, d, true))) return rc;
    hs[size_t(sub_index)].active = false;
    pkt_detach(ctx, hs[size_t(sub_index)]);
    const size_t nb_cifs = size_t(ctx->P.nb_cifs);
    for (size_t c = 0; c < nb_cifs; c++)
        CUDA_TRY(cudaMemset(ctx->d_msc_valid.as<uint8_t>() + (size_t(stream) * nb_cifs + c) * ctx->max_subs + size_t(sub_index), 0, 1));
    return upload_nsubs(ctx, stream, hs.size());
}

int dabgpu_softbits_push(dabgpu_ctx* ctx, const int8_t* frames_host, size_t stride, int first, int n) {
    int rc = check_stream_range(ctx, first, n);
    if (rc) return rc;
    if (!frames_host) return set_error(DABGPU_ERR_INVALID, "null frames");
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    // BasicRadio::Process requires exactly nb_frame_bits per call (basic_radio.cpp:41-46): the caller passes whole frames
    const size_t fb = size_t(ctx->P.nb_frame_bits);
    CUDA_TRY(sync_ctx(ctx));
    if ((rc = ctx->h_stage.alloc(size_t(n) * 8 + 64))) return rc;
    uint32_t* written = ctx->h_stage.as<uint32_t>();
    uint32_t* decoded = written + n;
    CUDA_TRY(cudaMemcpy(written, ctx->d_frames_written.as<uint32_t>() + first, size_t(n) * 4, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(decoded, ctx->d_frames_decoded.as<uint32_t>() + first, size_t(n) * 4, cudaMemcpyDeviceToHost));
    // the ring is full when one more frame would overwrite the history of the oldest undecoded one (the reference's
    // ThreadedRingBuffer blocks its producer there, src/radio_block.cpp:20-44): refuse instead of corrupting it
    for (int i = 0; i < n; i++)
        if (written[i] - decoded[i] >= ctx->chan.max_lag)
            return set_error(DABGPU_ERR_OVERFLOW, "soft-bit frame ring of stream %d is full (%u frames not channel-decoded yet): call dabgpu_chan_decode", first + i,
                             written[i] - decoded[i]);
    // natural-order frames -> staging -> ring layout (planar MSC); every stream writes the slot its counter points at
    if ((rc = ctx->d_pushstage.alloc(size_t(n) * fb))) return rc;
    CUDA_TRY(cudaMemcpy2DAsync(ctx->d_pushstage.p, fb, frames_host, stride, fb, size_t(n), cudaMemcpyHostToDevice, ctx->stream));
    k_frame_convert<<<dim3(16, n), 256, 0, ctx->stream>>>(ctx->d_pushstage.as<int8_t>(), fb, ctx->d_frames.as<int8_t>() + size_t(first) * ctx->frame_slots * fb,
                                                       size_t(ctx->frame_slots) * fb, ctx->d_frames_written.as<uint32_t>(), first, 0u, 0u, ctx->chan.geom, 1);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    for (int i = 0; i < n; i++) written[i] += 1;
    CUDA_TRY(cudaMemcpyAsync(ctx->d_frames_written.as<uint32_t>() + first, written, size_t(n) * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(sync_ctx(ctx));
    return DABGPU_OK;
}

// ---------------------------------------------------------------------------------------------
// Capture file formats (host only)
// ---------------------------------------------------------------------------------------------
int dabgpu_iq_convert(const char* mode, const void* raw, size_t n_bytes, float* out_c32, size_t out_cap_floats, size_t* n_floats) {
    if (!mode || (!raw && n_bytes) || !out_c32 || !n_floats) return set_error(DABGPU_ERR_INVALID, "null argument");
    const int fmt = dabgpu_host::iq_format_from_mode(mode);
    if (fmt < 0) return set_error(DABGPU_ERR_INVALID, "Unknown iq file format: '%s'", mode);
    const size_t n = n_bytes / dabgpu_host::iq_component_bytes(fmt);
    if (n > out_cap_floats) return set_error(DABGPU_ERR_OVERFLOW, "%zu components, room for %zu", n, out_cap_floats);
    *n_floats = dabgpu_host::iq_convert_to_c32(fmt, static_cast<const uint8_t*>(raw), n_bytes, out_c32);
    return DABGPU_OK;
}

int dabgpu_softbits_to_bytes(const int8_t* bits, size_t n_bits, uint8_t* bytes) {
    if (!bits || !bytes) return set_error(DABGPU_ERR_INVALID, "null argument");
    if (n_bits % 8) return set_error(DABGPU_ERR_INVALID, "%zu soft bits are not a whole number of bytes", n_bits);
    dabgpu_host::softbits_to_hard_bytes(bits, n_bits / 8, bytes);
    return DABGPU_OK;
}

int dabgpu_bytes_to_softbits(const uint8_t* bytes, size_t n_bytes, int8_t* bits) {
    if (!bits || !bytes) return set_error(DABGPU_ERR_INVALID, "null argument");
    dabgpu_host::hard_bytes_to_softbits(bytes, n_bytes, bits);
    return DABGPU_OK;
}

// ---------------------------------------------------------------------------------------------
// Self-configuration from the FIC (host only)
// ---------------------------------------------------------------------------------------------
struct dabgpu_autocfg {
    dabgpu_host::FIC_Autoconfig db;
    std::vector<uint8_t> applied_ids;    // SubChIds that got a decoder, in sub_index order
    std::vector<uint8_t> rejected_ids;   // complete in the database but not decodable (bad range / protection profile): never retried
};

dabgpu_autocfg* dabgpu_autocfg_create(void) { return new dabgpu_autocfg(); }
void dabgpu_autocfg_destroy(dabgpu_autocfg* a) { delete a; }

int dabgpu_autocfg_push_fibs(dabgpu_autocfg* a, const uint8_t* fibs, int n_fibs, size_t stride, const uint8_t* crc_ok) {
    if (!a || (!fibs && n_fibs > 0)) return set_error(DABGPU_ERR_INVALID, "null argument");
    if (stride < 30) return set_error(DABGPU_ERR_INVALID, "FIB stride %zu < 30", stride);
    int changed = 0;
    for (int i = 0; i < n_fibs; i++) {
        if (crc_ok && !crc_ok[i]) continue;   // FIC_Decoder only emits FIBs whose CRC matched (fic_decoder.cpp:98-116)
        if (a->db.ProcessFIB(fibs + size_t(i) * stride, 30)) changed++;
    }
    return changed;
}

int dabgpu_autocfg_dump(dabgpu_autocfg* a, int32_t* subs, int subs_cap_rows, int* n_subs, int32_t* comps, int comps_cap_rows, int* n_comps) {
    if (!a || !n_subs || !n_comps) return set_error(DABGPU_ERR_INVALID, "null argument");
    const auto& S = a->db.subchannels();
    const auto& Cc = a->db.components();
    *n_subs = int(S.size());
    *n_comps = int(Cc.size());
    if ((subs && subs_cap_rows < *n_subs) || (comps && comps_cap_rows < *n_comps)) return set_error(DABGPU_ERR_OVERFLOW, "dump buffers too small");
    if (subs)
        for (size_t i = 0; i < S.size(); i++) {
            const int32_t row[DABGPU_AUTOCFG_SUB_COLS] = {S[i].id, S[i].start_address, S[i].length, S[i].is_uep, S[i].uep_prot_index, S[i].eep_prot_level,
                                                         S[i].eep_type, S[i].fec_scheme, S[i].is_complete};
            memcpy(subs + i * DABGPU_AUTOCFG_SUB_COLS, row, sizeof(row));
        }
    if (comps)
        for (size_t i = 0; i < Cc.size(); i++) {
            const int32_t row[DABGPU_AUTOCFG_COMP_COLS] = {int32_t(Cc[i].service_value), Cc[i].service_type, Cc[i].component_id, Cc[i].subchannel_id, Cc[i].global_id,
                                                          Cc[i].transport_mode, Cc[i].audio_type, Cc[i].data_type, Cc[i].packet_address, Cc[i].is_complete};
            memcpy(comps + i * DABGPU_AUTOCFG_COMP_COLS, row, sizeof(row));
        }
    return DABGPU_OK;
}

int dabgpu_autocfg_runnable(dabgpu_autocfg* a, dabgpu_subchannel* out, uint8_t* ids, int cap, int* n_out) {
    if (!a || !n_out) return set_error(DABGPU_ERR_INVALID, "null argument");
    std::vector<dabgpu_subchannel> v;
    std::vector<uint8_t> id;
    a->db.Runnable(v, id);
    *n_out = int(v.size());
    if (out || ids) {
        if (cap < *n_out) return set_error(DABGPU_ERR_OVERFLOW, "%d runnable sub-channels, room for %d", *n_out, cap);
        for (size_t i = 0; i < v.size(); i++) { if (out) out[i] = v[i]; if (ids) ids[i] = id[i]; }
    }
    return DABGPU_OK;
}

// BasicRadio::UpdateAfterProcessing (basic_radio.cpp:83-154): every sub-channel that became runnable since the last call gets a
// decoder (dabgpu_msc_add_subchannel); the running ones are not touched.  A sub-channel the context refuses (range or
// protection profile invalid) is remembered and skipped: in the reference a bad sub-channel only affects itself.
// One dabgpu_autocfg object serves one (context, stream) pair whose table it fills alone.
int dabgpu_autocfg_apply(dabgpu_autocfg* a, dabgpu_ctx* ctx, int stream) {
    if (!a || !ctx) return set_error(DABGPU_ERR_INVALID, "null argument");
    std::vector<dabgpu_subchannel> v;
    std::vector<uint8_t> id;
    a->db.Runnable(v, id);
    int added = 0;
    for (size_t i = 0; i < v.size(); i++) {
        if (std::find(a->applied_ids.begin(), a->applied_ids.end(), id[i]) != a->applied_ids.end()) continue;
        if (std::find(a->rejected_ids.begin(), a->rejected_ids.end(), id[i]) != a->rejected_ids.end()) continue;
        const int rc = dabgpu_msc_add_subchannel(ctx, stream, &v[i], nullptr);
        if (rc == DABGPU_ERR_INVALID || rc == DABGPU_ERR_OVERFLOW) { a->rejected_ids.push_back(id[i]); continue; }
        if (rc) return rc;
        a->applied_ids.push_back(id[i]);
        added++;
    }
    return added > 0 ? 1 : 0;
}

int dabgpu_autocfg_applied(dabgpu_autocfg* a, uint8_t* ids, int cap, int* n_out) {
    if (!a || !n_out) return set_error(DABGPU_ERR_INVALID, "null argument");
    *n_out = int(a->applied_ids.size());
    if (ids) {
        if (cap < *n_out) return set_error(DABGPU_ERR_OVERFLOW, "%d applied sub-channels, room for %d", *n_out, cap);
        memcpy(ids, a->applied_ids.data(), a->applied_ids.size());
    }
    return DABGPU_OK;
}

// The packet entries of every stream, by stream then index, on the host and (queued on ctx->stream) on the device.  Rebuilt when
// the sub-channel tables change (cfg_epoch); every table change first synchronises the context, so nothing queued still reads
// the old device copy then.
static int pkt_items(dabgpu_ctx* ctx) {
    PacketState& P = ctx->packet;
    if (P.items_epoch == ctx->cfg_epoch) return DABGPU_OK;
    P.items.clear();
    for (size_t s = 0; s < ctx->subs.size(); s++)
        for (size_t k = 0; k < ctx->subs[s].size(); k++) {
            const SubHost& h = ctx->subs[s][k];
            if (h.active && h.is_packet()) P.items.push_back(PktItemDev{uint32_t(s), uint32_t(k), uint64_t(h.pkt_region)});
        }
    if (!P.items.empty()) {
        int rc;
        if ((rc = P.d_items.alloc(P.items.size() * sizeof(PktItemDev)))) return rc;
        CUDA_TRY(cudaMemcpyAsync(P.d_items.p, P.items.data(), P.items.size() * sizeof(PktItemDev), cudaMemcpyHostToDevice, ctx->stream));
    }
    P.items_epoch = ctx->cfg_epoch;
    return DABGPU_OK;
}

// The kernels of one channel decode, all on ctx->stream (which dabgpu_chan_decode points at the channel stream meanwhile).
static int chan_decode_body(dabgpu_ctx* ctx, int first, int n) {
    int rc;
    const uint32_t total = uint32_t(n) * ctx->chan.jobs_per_stream;
    if ((rc = ctx->d_jobs.alloc(size_t(total) * sizeof(VitJobDev)))) return rc;
    VlPlan* count_plan = (ctx->vl_mode != 2) ? ctx->d_vlplan.as<VlPlan>() : nullptr;
    ctx->prof.begin(PROF_CHAN_MISC, ctx->stream);
    if (count_plan) CUDA_TRY(cudaMemsetAsync(count_plan, 0, sizeof(VlPlan), ctx->stream));
    k_chan_build_jobs<<<(total + 127) / 128, 128, 0, ctx->stream>>>(ctx->chan, ctx->d_jobs.as<VitJobDev>(), first, n, count_plan);
    {
        const uint32_t cus = uint32_t(ctx->P.nb_cif_bits) / 64u;
        k_chan_deinterleave<<<dim3((cus + 287u) / 288u, uint32_t(n) * uint32_t(ctx->P.nb_cifs)), 288, 0, ctx->stream>>>(ctx->chan, first);
    }
    ctx->prof.end(ctx->stream);
    ctx->launches += 2;
    if (ctx->vl_cache.first != first || ctx->vl_cache.n != n || ctx->vl_cache.epoch != ctx->cfg_epoch) {
        VlBound vb;
        ctx->vl_cache.max_subs_used = 0;
        for (int s = first; s < first + n; s++) {
            ctx->vl_cache.max_subs_used = std::max(ctx->vl_cache.max_subs_used, uint32_t(ctx->subs[size_t(s)].size()));
            if (ctx->chan.fic_enabled) vb.add(774u, uint32_t(ctx->P.nb_cifs));
            for (const SubHost& h : ctx->subs[size_t(s)]) if (h.active) vb.add(uint32_t(h.sched.total_steps()), uint32_t(ctx->P.nb_cifs));
        }
        memcpy(ctx->vl_cache.count, vb.count, sizeof(vb.count));
        ctx->vl_cache.max_steps = vb.max_steps;
        ctx->vl_cache.first = first; ctx->vl_cache.n = n; ctx->vl_cache.epoch = ctx->cfg_epoch;
    }
    {
        VlBound vb;
        memcpy(vb.count, ctx->vl_cache.count, sizeof(vb.count));
        vb.max_steps = ctx->vl_cache.max_steps;
        if ((rc = launch_viterbi(ctx, ctx->d_jobs.as<VitJobDev>(), int(total), &vb, count_plan != nullptr))) return rc;
    }
    if ((rc = dabplus_run(ctx->dabplus, ctx->chan, first, n, ctx->vl_cache.max_subs_used, ctx->num_sms, ctx->stream, &ctx->launches, ctx->prof))) return rc;
    if ((rc = pkt_items(ctx))) return rc;
    if ((rc = packet_run(ctx->packet, ctx->chan, first, n, ctx->num_sms, ctx->stream, &ctx->launches, ctx->prof))) return rc;
    ctx->prof.begin(PROF_CHAN_MISC, ctx->stream);
    k_chan_finish<<<n, 32, 0, ctx->stream>>>(ctx->chan, first, n);
    ctx->prof.end(ctx->stream);
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    return DABGPU_OK;
}

// The channel decode of a step runs on its own CUDA stream so that it overlaps whatever the caller queues next on the main
// stream -- in a receiver loop the OFDM stage of the next step.  The lane Viterbi leaves half of every sub-partition's issue
// slots empty at 256 streams and the OFDM kernels are latency bound, so the two fill each other's gaps.  Hazards: the OFDM
// stage writes the frame-ring slot of frame n+1 while the decode of frame n reads the slots n-4..n (the ring keeps two frames
// of margin, see frame_slots); every other buffer of the channel decode is only touched on the channel stream.  The main
// stream joins (join_dabplus) before the next channel decode -- which bounds the lead to one step --, before every
// synchronising getter, before dabgpu_viterbi_decode / dabgpu_fic_decode (shared job and scratch buffers) and before the
// pipeline's compute-done event.  While profiling, everything stays on the main stream.
int dabgpu_chan_decode(dabgpu_ctx* ctx, int first, int n) {
    int rc = check_stream_range(ctx, first, n);
    if (rc) return rc;
    if (n == 0) return DABGPU_OK;
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(join_dabplus(ctx));
    const bool fork = ctx->s_dp != nullptr && !ctx->prof.on;
    cudaStream_t main_stream = ctx->stream;
    // what the OFDM stage (or dabgpu_softbits_push) has produced so far; the decode kernels only read this copy, because the
    // next OFDM stage advances the live counters on the main stream while the decode runs on the channel stream
    CUDA_TRY(cudaMemcpyAsync(ctx->d_frames_snapshot.as<uint32_t>() + first, ctx->d_frames_written.as<uint32_t>() + first, size_t(n) * 4,
                             cudaMemcpyDeviceToDevice, main_stream));
    if (fork) {
        CUDA_TRY(cudaEventRecord(ctx->ev_dp_fork, main_stream));
        CUDA_TRY(cudaStreamWaitEvent(ctx->s_dp, ctx->ev_dp_fork, 0));
        ctx->stream = ctx->s_dp;
    }
    rc = chan_decode_body(ctx, first, n);
    if (fork) {
        ctx->stream = main_stream;
        if (cudaEventRecord(ctx->ev_dp, ctx->s_dp) == cudaSuccess) ctx->dp_pending = true;
    }
    return rc;
}

// Non-blocking: everything queued on the context's stream after this call waits for the last dabgpu_chan_decode.
int dabgpu_chan_join(dabgpu_ctx* ctx) {
    if (!ctx) return set_error(DABGPU_ERR_INVALID, "null context");
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(join_dabplus(ctx));
    return DABGPU_OK;
}

int dabgpu_chan_get_status(dabgpu_ctx* ctx, int stream, dabgpu_chan_status* out) {
    int rc = check_stream_range(ctx, stream, 1);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(sync_ctx(ctx));
    int32_t st[2];
    CUDA_TRY(cudaMemcpy(st, ctx->d_status.as<int32_t>() + 2 * stream, 8, cudaMemcpyDeviceToHost));
    out->decoded = st[0];
    out->frame_index = st[1];
    return DABGPU_OK;
}

int dabgpu_chan_get_fic(dabgpu_ctx* ctx, int stream, uint8_t* fibs_host, uint8_t* crc_ok) {
    int rc = check_stream_range(ctx, stream, 1);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(sync_ctx(ctx));
    const int nb_cifs = ctx->P.nb_cifs, nf = ctx->P.nb_fibs_per_cif;
    std::vector<uint8_t> tmp(size_t(nb_cifs) * FIC_GROUP_BYTES), crc(size_t(nb_cifs) * 4);
    CUDA_TRY(cudaMemcpy(tmp.data(), ctx->d_fic_out.as<uint8_t>() + size_t(stream) * nb_cifs * FIC_GROUP_BYTES, tmp.size(), cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(crc.data(), ctx->d_fic_crc.as<uint8_t>() + size_t(stream) * nb_cifs * 4, crc.size(), cudaMemcpyDeviceToHost));
    for (int c = 0; c < nb_cifs; c++) {
        if (fibs_host) memcpy(fibs_host + size_t(c) * nf * 32, tmp.data() + size_t(c) * FIC_GROUP_BYTES, size_t(nf) * 32);
        if (crc_ok) for (int f = 0; f < nf; f++) crc_ok[c * nf + f] = ctx->chan.fic_enabled ? crc[size_t(c) * 4 + f] : 0;
    }
    return DABGPU_OK;
}

int dabgpu_chan_get_msc(dabgpu_ctx* ctx, int stream, int sub_index, uint8_t* out_host, size_t out_cap, uint8_t* valid, int* bytes_per_cif) {
    int rc = check_stream_range(ctx, stream, 1);
    if (rc) return rc;
    const auto& hs = ctx->subs[size_t(stream)];
    if (sub_index < 0 || size_t(sub_index) >= hs.size() || !hs[size_t(sub_index)].active) return set_error(DABGPU_ERR_INVALID, "sub-channel index %d not configured", sub_index);
    const SubHost& h = hs[size_t(sub_index)];
    const int nb_cifs = ctx->P.nb_cifs;
    if (bytes_per_cif) *bytes_per_cif = int(h.n_out_bytes);
    if (out_host && out_cap < size_t(nb_cifs) * h.n_out_bytes) return set_error(DABGPU_ERR_OVERFLOW, "output buffer too small");
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(sync_ctx(ctx));
    for (int c = 0; c < nb_cifs; c++) {
        if (out_host)
            CUDA_TRY(cudaMemcpy(out_host + size_t(c) * h.n_out_bytes,
                                ctx->d_msc_out.as<uint8_t>() + (size_t(stream) * nb_cifs + c) * CIF_OUT_STRIDE + h.out_offset, h.n_out_bytes,
                                cudaMemcpyDeviceToHost));
        if (valid)
            CUDA_TRY(cudaMemcpy(valid + c, ctx->d_msc_valid.as<uint8_t>() + (size_t(stream) * nb_cifs + c) * ctx->max_subs + sub_index, 1,
                                cudaMemcpyDeviceToHost));
    }
    return DABGPU_OK;
}

int dabgpu_chan_get_dabplus_events(dabgpu_ctx* ctx, int stream, int sub_index, uint8_t* log_host, size_t log_cap, size_t* log_bytes) {
    int rc = check_stream_range(ctx, stream, 1);
    if (rc) return rc;
    if (sub_index < 0 || size_t(sub_index) >= ctx->subs[size_t(stream)].size() || !ctx->subs[size_t(stream)][size_t(sub_index)].active)
        return set_error(DABGPU_ERR_INVALID, "sub-channel index %d not configured", sub_index);
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(sync_ctx(ctx));
    const SubHost& h = ctx->subs[size_t(stream)][size_t(sub_index)];
    if (h.is_packet()) return packet_get_events(ctx->packet, uint64_t(h.pkt_region), log_host, log_cap, log_bytes);
    return dabplus_get_events(ctx->dabplus, stream, sub_index, log_host, log_cap, log_bytes);
}

// The packed output layout over every stream: dp_pack_item_bound for each active DAB+ sub-channel, pkt_item_bound for each
// active packet entry, 0 for every other entry of the [max_streams][max_subs] table.  It depends only on the sub-channel tables and is rebuilt when they change
// (cfg_epoch).  Every table change first synchronises the context, so no queued pack still reads the device copy then.
static const std::vector<uint64_t>& dp_layout(dabgpu_ctx* ctx) {
    DabPlusState& D = ctx->dabplus;
    if (D.layout_epoch != ctx->cfg_epoch) {
        const size_t ms = size_t(ctx->max_subs);
        D.layout.assign(ctx->subs.size() * ms + 1, 0);
        uint64_t at = 0;
        for (size_t s = 0; s < ctx->subs.size(); s++)
            for (size_t k = 0; k < ms; k++) {
                D.layout[s * ms + k] = at;
                const SubHost* h = k < ctx->subs[s].size() ? &ctx->subs[s][k] : nullptr;
                if (h && h->active && h->sc.is_dabplus) at += dp_pack_item_bound(h->n_out_bytes);
                if (h && h->active && h->is_packet()) at += h->pkt_cap;
            }
        D.layout.back() = at;
        D.layout_epoch = ctx->cfg_epoch;
    }
    return D.layout;
}

// Log bytes one decode of streams [first, first + n) can produce; the index holds int32 offsets, so it must stay below 2^31.
static int dp_range_bound(dabgpu_ctx* ctx, int first, int n, size_t* bytes) {
    const std::vector<uint64_t>& lay = dp_layout(ctx);
    const uint64_t b = lay[size_t(first + n) * ctx->max_subs] - lay[size_t(first) * ctx->max_subs];
    if (b > uint64_t(INT32_MAX)) return set_error(DABGPU_ERR_INVALID, "DAB+ log of streams [%d,%d) may reach %llu bytes: use smaller ranges", first, first + n, (unsigned long long)b);
    *bytes = size_t(b);
    return DABGPU_OK;
}

// A DAB+ output request for streams [first, first + n), checked before anything is queued.
static int dp_check_out(dabgpu_ctx* ctx, int first, int n, const dabgpu_dabplus_out* out, size_t* log_bytes) {
    if (!out->log_host || !out->index_host) return set_error(DABGPU_ERR_INVALID, "null DAB+ log or index buffer");
    int rc = dp_range_bound(ctx, first, n, log_bytes);
    if (rc) return rc;
    if (out->log_cap < *log_bytes) return set_error(DABGPU_ERR_OVERFLOW, "DAB+ log buffer of %zu bytes, streams [%d,%d) need %zu (dabgpu_dabplus_out_bound)", out->log_cap, first, first + n, *log_bytes);
    return DABGPU_OK;
}

// Queues k_dabplus_pack on ctx->stream into d_buf: the log (log_bytes) first, the index at dp_index_offset(log_bytes).
static size_t dp_index_offset(size_t log_bytes) { return (log_bytes + 255u) & ~size_t(255); }
static int dp_pack(dabgpu_ctx* ctx, int first, int n, size_t log_bytes, DevBuf& d_buf) {
    DabPlusState& D = ctx->dabplus;
    const std::vector<uint64_t>& lay = dp_layout(ctx);
    int rc;
    if (D.layout_dev_epoch != D.layout_epoch) {
        if ((rc = D.d_layout.alloc(lay.size() * sizeof(uint64_t)))) return rc;
        CUDA_TRY(cudaMemcpyAsync(D.d_layout.p, lay.data(), lay.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
        D.layout_dev_epoch = D.layout_epoch;
    }
    const size_t at = dp_index_offset(log_bytes);
    if ((rc = d_buf.alloc(at + size_t(n) * ctx->max_subs * 8))) return rc;
    uint32_t subs_per_stream = 0;
    for (int s = first; s < first + n; s++) subs_per_stream = std::max(subs_per_stream, uint32_t(ctx->subs[size_t(s)].size()));
    if ((rc = dabplus_pack(D, first, n, subs_per_stream, d_buf.as<uint8_t>(), reinterpret_cast<int32_t*>(d_buf.as<uint8_t>() + at), ctx->stream,
                           &ctx->launches, ctx->prof)))
        return rc;
    // the packet entries' logs and index entries, over what k_dabplus_pack left empty for them
    if ((rc = pkt_items(ctx))) return rc;
    return packet_pack(ctx->packet, D.d_layout.as<uint64_t>(), first, n, ctx->max_subs, d_buf.as<uint8_t>(),
                       reinterpret_cast<int32_t*>(d_buf.as<uint8_t>() + at), ctx->stream, &ctx->launches, ctx->prof);
}

static int dp_copy_out(dabgpu_ctx* ctx, int n, size_t log_bytes, const DevBuf& d_buf, const dabgpu_dabplus_out* out, cudaStream_t s) {
    CUDA_TRY(cudaMemcpyAsync(out->log_host, d_buf.p, log_bytes, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(out->index_host, d_buf.as<uint8_t>() + dp_index_offset(log_bytes), size_t(n) * ctx->max_subs * 8, cudaMemcpyDeviceToHost, s));
    return DABGPU_OK;
}

int dabgpu_dabplus_out_bound(dabgpu_ctx* ctx, int first_stream, int n_streams, size_t* log_bytes) {
    int rc = check_stream_range(ctx, first_stream, n_streams);
    if (rc) return rc;
    if (!log_bytes) return set_error(DABGPU_ERR_INVALID, "null output");
    return dp_range_bound(ctx, first_stream, n_streams, log_bytes);
}

int dabgpu_chan_get_dabplus_all(dabgpu_ctx* ctx, int first_stream, int n_streams, const dabgpu_dabplus_out* out) {
    int rc = check_stream_range(ctx, first_stream, n_streams);
    if (rc) return rc;
    if (!out) return set_error(DABGPU_ERR_INVALID, "null DAB+ output");
    size_t log_bytes = 0;
    if ((rc = dp_check_out(ctx, first_stream, n_streams, out, &log_bytes))) return rc;
    if (n_streams == 0) return DABGPU_OK;
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(join_dabplus(ctx));
    if ((rc = dp_pack(ctx, first_stream, n_streams, log_bytes, ctx->dabplus.d_out))) return rc;
    if ((rc = dp_copy_out(ctx, n_streams, log_bytes, ctx->dabplus.d_out, out, ctx->stream))) return rc;
    CUDA_TRY(sync_ctx(ctx));
    return DABGPU_OK;
}

int dabgpu_rs_decode(dabgpu_ctx* ctx, uint8_t* codewords_host, int n_codewords, int nroots, int pad, int* counts_host, int* positions_host) {
    if (!ctx || !codewords_host || !counts_host) return set_error(DABGPU_ERR_INVALID, "null argument");
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(join_dabplus(ctx));
    return dabplus_rs_decode_batch(ctx->dabplus, codewords_host, n_codewords, nroots, pad, counts_host, positions_host, ctx->stream, &ctx->launches);
}

int dabgpu_packet_fec_decode(dabgpu_ctx* ctx, uint8_t* frames_host, int n_frames, int* row_counts_host) {
    if (!ctx || !frames_host) return set_error(DABGPU_ERR_INVALID, "null argument");
    if (n_frames < 0) return set_error(DABGPU_ERR_INVALID, "n_frames %d", n_frames);
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(join_dabplus(ctx));
    return dabplus_packet_fec_batch(ctx->dabplus, frames_host, n_frames, row_counts_host, ctx->stream, &ctx->launches);
}

int dabgpu_fic_decode(dabgpu_ctx* ctx, const int8_t* soft_host, int n_groups, uint8_t* fibs_host, uint8_t* crc_ok) {
    if (!ctx || !soft_host || !fibs_host || !crc_ok) return set_error(DABGPU_ERR_INVALID, "null argument");
    if (n_groups <= 0) return DABGPU_OK;
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(join_dabplus(ctx));
    int rc;
    const size_t n = size_t(n_groups);
    if ((rc = ctx->d_vsoft.alloc(n * 2304 + 1024))) return rc;
    if ((rc = ctx->d_vout.alloc(n * (FIC_GROUP_BYTES + 4) + 16))) return rc;
    if ((rc = ctx->d_jobs.alloc(n * sizeof(VitJobDev)))) return rc;
    std::vector<VitJobDev> hj(n);
    uint8_t* d_crc = ctx->d_vout.as<uint8_t>() + n * FIC_GROUP_BYTES;
    for (size_t i = 0; i < n; i++) {
        VitJobDev& J = hj[i];
        memset(&J, 0, sizeof(J));
        // PI_16 x 21 blocks, PI_15 x 3 blocks, tail (fic_decoder.cpp:74-85)
        J.src = ctx->d_vsoft.as<int8_t>() + i * 2304;
        J.out = ctx->d_vout.as<uint8_t>() + i * FIC_GROUP_BYTES;
        J.crc_ok = d_crc + i * 4;
        J.seg_pi[0] = 16; J.seg_pi[1] = 15; J.seg_pi[2] = 0;
        J.seg_step_end[0] = 672; J.seg_step_end[1] = 768; J.seg_step_end[2] = 774; J.seg_step_end[3] = 774; J.seg_step_end[4] = 774;
        J.seg_in_base[0] = 0; J.seg_in_base[1] = 2016; J.seg_in_base[2] = 2292;
        J.n_seg = 3; J.total_steps = 774; J.n_out_bytes = 96;
        J.flags = VJ_DESCRAMBLE | VJ_FIB_CRC;
        J.n_fibs = 3;
    }
    CUDA_TRY(cudaMemcpyAsync(ctx->d_vsoft.p, soft_host, n * 2304, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(ctx->d_jobs.p, hj.data(), n * sizeof(VitJobDev), cudaMemcpyHostToDevice, ctx->stream));
    {
        VlBound vb;
        vb.add(774u, uint32_t(n_groups));
        if ((rc = launch_viterbi(ctx, ctx->d_jobs.as<VitJobDev>(), n_groups, &vb))) return rc;
    }
    std::vector<uint8_t> tmp(n * (FIC_GROUP_BYTES + 4));
    CUDA_TRY(cudaMemcpyAsync(tmp.data(), ctx->d_vout.p, tmp.size(), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(sync_ctx(ctx));
    for (size_t i = 0; i < n; i++) {
        memcpy(fibs_host + i * 96, tmp.data() + i * FIC_GROUP_BYTES, 96);
        memcpy(crc_ok + i * 3, tmp.data() + n * FIC_GROUP_BYTES + i * 4, 3);
    }
    return DABGPU_OK;
}

struct dabgpu_dabplus { DabPlusProc* d = nullptr; };

int dabgpu_dabplus_open(dabgpu_ctx* ctx, dabgpu_dabplus** out) {
    if (!ctx || !out) return set_error(DABGPU_ERR_INVALID, "null argument");
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    dabgpu_dabplus* p = new dabgpu_dabplus();
    cudaError_t e = cudaMalloc(&p->d, sizeof(DabPlusProc));
    if (e != cudaSuccess) { delete p; return set_error(DABGPU_ERR_NOMEM, "cudaMalloc: %s", cudaGetErrorString(e)); }
    cudaMemset(p->d, 0, sizeof(DabPlusProc));
    *out = p;
    return DABGPU_OK;
}

void dabgpu_dabplus_close(dabgpu_ctx* ctx, dabgpu_dabplus* p) {
    if (!p) return;
    if (ctx) { cudaSetDevice(ctx->cfg.device); sync_ctx(ctx); }
    if (p->d) cudaFree(p->d);
    delete p;
}

int dabgpu_dabplus_process(dabgpu_ctx* ctx, dabgpu_dabplus* p, const uint8_t* frame_host, int n_bytes, uint8_t* log_host, size_t log_cap, size_t* log_bytes) {
    if (!ctx || !p || !frame_host) return set_error(DABGPU_ERR_INVALID, "null argument");
    if (n_bytes < 0 || n_bytes > int(CIF_OUT_STRIDE)) return set_error(DABGPU_ERR_INVALID, "logical frame of %d bytes out of range", n_bytes);
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(cudaMemcpyAsync(p->d->frame, frame_host, size_t(n_bytes), cudaMemcpyHostToDevice, ctx->stream));
    k_dabplus_direct<<<1, 32, 0, ctx->stream>>>(p->d, n_bytes, ctx->d_counters.as<unsigned long long>());
    ctx->launches++;
    CUDA_TRY(cudaGetLastError());
    int32_t n_ev = 0;
    CUDA_TRY(cudaMemcpyAsync(&n_ev, &p->d->n_events, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(sync_ctx(ctx));
    if (n_ev > DP_MAX_EVENTS) return set_error(DABGPU_ERR_OVERFLOW, "event queue overflow (%d events)", n_ev);
    DabPlusEvent ev[DP_MAX_EVENTS];
    if (n_ev > 0) CUDA_TRY(cudaMemcpy(ev, p->d->events, size_t(n_ev) * sizeof(DabPlusEvent), cudaMemcpyDeviceToHost));
    size_t off = 0;
    for (int i = 0; i < n_ev; i++) {
        const size_t padded = (size_t(ev[i].payload_len) + 3u) & ~size_t(3);
        if (off + 24 + padded > log_cap) return set_error(DABGPU_ERR_OVERFLOW, "event log buffer too small");
        const int32_t hdr[6] = {ev[i].type, ev[i].a, ev[i].b, ev[i].c, ev[i].d, ev[i].payload_len};
        if (log_host) memcpy(log_host + off, hdr, 24);
        off += 24;
        if (ev[i].payload_len > 0) {
            if (log_host) {
                memset(log_host + off, 0, padded);
                CUDA_TRY(cudaMemcpy(log_host + off, p->d->sf_out + ev[i].payload_off, size_t(ev[i].payload_len), cudaMemcpyDeviceToHost));
            }
            off += padded;
        }
    }
    if (log_bytes) *log_bytes = off;
    return DABGPU_OK;
}

int dabgpu_get_counters(dabgpu_ctx* ctx, dabgpu_counters* out) {
    if (!ctx || !out) return set_error(DABGPU_ERR_INVALID, "null argument");
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(sync_ctx(ctx));
    unsigned long long c[CNT_COUNT];
    CUDA_TRY(cudaMemcpy(c, ctx->d_counters.p, sizeof(c), cudaMemcpyDeviceToHost));
    out->frames_demodulated = c[CNT_FRAMES_DEMOD];
    out->frames_channel_decoded = c[CNT_FRAMES_CHAN];
    out->fibs_crc_ok = c[CNT_FIB_OK];
    out->fibs_total = c[CNT_FIB_TOTAL];
    out->msc_bytes_decoded = c[CNT_MSC_BYTES];
    out->superframes_ok = c[CNT_SF_OK];
    out->superframes_rs_fail = c[CNT_SF_RS_FAIL];
    out->superframes_firecode_fail = c[CNT_SF_FIRE_FAIL];
    out->au_ok = c[CNT_AU_OK];
    out->au_crc_fail = c[CNT_AU_CRC_FAIL];
    out->frames_dropped = c[CNT_FRAMES_DROPPED];
    return DABGPU_OK;
}

// ---------------------------------------------------------------------------------------------
// OFDM (implementation in ofdm.cuh)
// ---------------------------------------------------------------------------------------------
int dabgpu_ofdm_set_config(dabgpu_ctx* ctx, const dabgpu_ofdm_config* cfg) {
    if (!ctx || !cfg) return set_error(DABGPU_ERR_INVALID, "null argument");
    if (int rc = validate_ofdm_config(*cfg)) return rc;
    ctx->cfg.ofdm = *cfg;
    ctx->ofdm.dev.cfg = *cfg;   // OfdmDev travels by value with every launch: the next call sees the new knobs
    return DABGPU_OK;
}

int dabgpu_ofdm_reset(dabgpu_ctx* ctx, int stream) {
    if (!ctx) return set_error(DABGPU_ERR_INVALID, "null context");
    if (stream < -1 || stream >= ctx->cfg.max_streams) return set_error(DABGPU_ERR_INVALID, "stream %d out of range", stream);
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    return ofdm_reset(ctx->ofdm, stream, ctx->stream);
}

// A channel decode that is still running on the channel stream reads frame-ring slots that the OFDM stage may overwrite once it
// emits more than two further frames (ChanDev.max_lag keeps two slots of margin): such calls wait for the decode first.
static cudaError_t join_if_many_frames(dabgpu_ctx* ctx, long n_samples) {
    const long max_frames = n_samples / long(ctx->P.nb_frame_samples - ctx->P.nb_cyclic_prefix) + 1;
    return (ctx->dp_pending && max_frames > 2) ? join_dabplus(ctx) : cudaSuccess;
}

int dabgpu_ofdm_process(dabgpu_ctx* ctx, const void* iq_host, size_t stride_bytes, int first, int n, int n_samples, int block_size) {
    int rc = check_stream_range(ctx, first, n);
    if (rc) return rc;
    if (!iq_host || n_samples < 0) return set_error(DABGPU_ERR_INVALID, "bad IQ buffer");
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(join_if_many_frames(ctx, n_samples));
    ctx->ofdm.demod_ctas_cap = ctx->dp_pending ? 3 : 0;   // a channel decode is running on its stream: share the SMs with it
    return ofdm_process(ctx->ofdm, iq_host, stride_bytes, first, n, n_samples, block_size, ctx->stream);
}

int dabgpu_ofdm_attach_device_input(dabgpu_ctx* ctx, const void* d_iq, size_t stride_samples, size_t capacity) {
    if (!ctx || !d_iq) return set_error(DABGPU_ERR_INVALID, "null argument");
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    return ofdm_attach(ctx->ofdm, d_iq, stride_samples, capacity, ctx->stream);
}

int dabgpu_ofdm_advance(dabgpu_ctx* ctx, int first, int n, int n_samples, int block_size) {
    int rc = check_stream_range(ctx, first, n);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(join_if_many_frames(ctx, n_samples));
    ctx->ofdm.demod_ctas_cap = ctx->dp_pending ? 3 : 0;   // a channel decode is running on its stream: share the SMs with it
    return ofdm_advance(ctx->ofdm, first, n, n_samples, block_size, ctx->stream);
}

int dabgpu_ofdm_get_response(dabgpu_ctx* ctx, int stream, int kind, float* out, int n_floats) {
    int rc = check_stream_range(ctx, stream, 1);
    if (rc) return rc;
    if (!out || kind < 0 || kind > 1) return set_error(DABGPU_ERR_INVALID, "bad argument");
    if (!ctx->ofdm.d_diag.p) return set_error(DABGPU_ERR_STATE, "context was created without DABGPU_FLAG_DIAG_TAPS");
    if (n_floats < ctx->P.nb_fft) return set_error(DABGPU_ERR_OVERFLOW, "response needs %d floats", ctx->P.nb_fft);
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(sync_ctx(ctx));
    CUDA_TRY(cudaMemcpy(out, ctx->ofdm.d_diag.as<float>() + (size_t(stream) * 2 + size_t(kind)) * size_t(ctx->P.nb_fft), size_t(ctx->P.nb_fft) * sizeof(float),
                        cudaMemcpyDeviceToHost));
    return DABGPU_OK;
}

int dabgpu_ofdm_get_correlation_buffer(dabgpu_ctx* ctx, int stream, float* out, size_t n_floats) {
    int rc = check_stream_range(ctx, stream, 1);
    if (rc) return rc;
    if (!out) return set_error(DABGPU_ERR_INVALID, "null output");
    const size_t n = size_t(ctx->P.nb_null_period + ctx->P.nb_symbol_period);
    if (n_floats < 2 * n) return set_error(DABGPU_ERR_OVERFLOW, "correlation buffer needs %zu floats", 2 * n);
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    CUDA_TRY(cudaMemcpy(out, ctx->ofdm.dev.corr + size_t(stream) * n, n * sizeof(float2), cudaMemcpyDeviceToHost));
    return DABGPU_OK;
}

int dabgpu_ofdm_get_frame_fft(dabgpu_ctx* ctx, int stream, float* out, size_t n_floats) {
    int rc = check_stream_range(ctx, stream, 1);
    if (rc) return rc;
    if (!out) return set_error(DABGPU_ERR_INVALID, "null output");
    const size_t need = size_t(ctx->P.nb_frame_symbols) * size_t(ctx->P.nb_fft) * 2;
    if (n_floats < need) return set_error(DABGPU_ERR_OVERFLOW, "frame spectrum needs %zu floats", need);
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(join_dabplus(ctx));
    // callers that give room for nb_frame_symbols + 1 rows also get the NULL-symbol row, like the reference's buffer
    const bool with_null = n_floats >= need + size_t(ctx->P.nb_fft) * 2;
    return ofdm_frame_fft(ctx->ofdm, stream, out, with_null, nullptr, ctx->stream);
}

int dabgpu_ofdm_get_frame_data_vec(dabgpu_ctx* ctx, int stream, float* out, size_t n_floats) {
    int rc = check_stream_range(ctx, stream, 1);
    if (rc) return rc;
    if (!out) return set_error(DABGPU_ERR_INVALID, "null output");
    const size_t need = size_t(ctx->P.nb_frame_symbols - 1) * size_t(ctx->P.nb_data_carriers) * 2;
    if (n_floats < need) return set_error(DABGPU_ERR_OVERFLOW, "frame data vectors need %zu floats", need);
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(join_dabplus(ctx));
    return ofdm_frame_fft(ctx->ofdm, stream, nullptr, false, out, ctx->stream);
}

int dabgpu_ofdm_get_status(dabgpu_ctx* ctx, int stream, dabgpu_ofdm_status* out) {
    int rc = check_stream_range(ctx, stream, 1);
    if (rc) return rc;
    if (!out) return set_error(DABGPU_ERR_INVALID, "null output");
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    rc = ofdm_get_status(ctx->ofdm, stream, out, ctx->stream);
    if (rc) return rc;
    uint32_t written = 0;
    CUDA_TRY(cudaMemcpy(&written, ctx->d_frames_written.as<uint32_t>() + stream, 4, cudaMemcpyDeviceToHost));
    out->frames_queued = int(written - ctx->h_frames_popped[size_t(stream)]);
    out->frames_dropped = int(ctx->h_frames_dropped[size_t(stream)]);
    return DABGPU_OK;
}

int dabgpu_ofdm_pop_frames(dabgpu_ctx* ctx, int stream, int8_t* frames_host, int max_frames, dabgpu_frame_info* infos, int* n_out) {
    int rc = check_stream_range(ctx, stream, 1);
    if (rc) return rc;
    if (!n_out) return set_error(DABGPU_ERR_INVALID, "null output");
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(sync_ctx(ctx));
    uint32_t written = 0;
    CUDA_TRY(cudaMemcpy(&written, ctx->d_frames_written.as<uint32_t>() + stream, 4, cudaMemcpyDeviceToHost));
    uint32_t& popped = ctx->h_frames_popped[size_t(stream)];
    // frames older than the ring depth were overwritten: the observer model of the reference drops nothing, so
    // callers must pop at least every frame_slots-2 frames; report the overrun instead of returning stale data
    if (written - popped > uint32_t(ctx->frame_slots - 1)) {
        ctx->h_frames_dropped[size_t(stream)] += (written - uint32_t(ctx->frame_slots - 1)) - popped;   // dabgpu_ofdm_status.frames_dropped
        popped = written - uint32_t(ctx->frame_slots - 1);
    }
    const size_t fb = size_t(ctx->P.nb_frame_bits);
    int n = 0;
    while (popped < written && n < max_frames) {
        const size_t slot = popped & uint32_t(ctx->frame_slots - 1);
        if (frames_host) {
            if ((rc = ctx->d_popstage.alloc(fb))) return rc;
            k_frame_convert<<<dim3(16, 1), 256, 0, ctx->stream>>>(ctx->d_popstage.as<int8_t>(), fb, ctx->d_frames.as<int8_t>() + size_t(stream) * ctx->frame_slots * fb,
                                                               size_t(ctx->frame_slots) * fb, nullptr, 0, 0u, uint32_t(slot), ctx->chan.geom, 0);
            ctx->launches++;
            CUDA_TRY(cudaGetLastError());
            CUDA_TRY(cudaMemcpyAsync(frames_host + size_t(n) * fb, ctx->d_popstage.p, fb, cudaMemcpyDeviceToHost, ctx->stream));
            CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        }
        if (infos)
            CUDA_TRY(cudaMemcpy(infos + n, ctx->d_frame_info.as<dabgpu_frame_info>() + size_t(stream) * ctx->frame_slots + slot, sizeof(dabgpu_frame_info), cudaMemcpyDeviceToHost));
        popped++;
        n++;
    }
    *n_out = n;
    return DABGPU_OK;
}

int dabgpu_ofdm_fetch_latest(dabgpu_ctx* ctx, int first, int n, int8_t* frames_host, uint8_t* produced) {
    int rc = check_stream_range(ctx, first, n);
    if (rc) return rc;
    if (!frames_host || !produced) return set_error(DABGPU_ERR_INVALID, "null output");
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    return ofdm_fetch_latest(ctx->ofdm, first, n, frames_host, produced, ctx->stream);
}

// ---------------------------------------------------------------------------------------------
// Pipelined step: H2D (copy stream) -> OFDM [+ channel decode] (compute stream) -> D2H (copy-out stream)
// ---------------------------------------------------------------------------------------------
static int pipe_init(dabgpu_ctx* ctx) {
    if (ctx->s_h2d) return DABGPU_OK;
    CUDA_TRY(cudaStreamCreateWithFlags(&ctx->s_h2d, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&ctx->s_d2h, cudaStreamNonBlocking));
    for (auto& sl : ctx->pipe) {
        CUDA_TRY(cudaEventCreateWithFlags(&sl.h2d_done, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&sl.compute_done, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&sl.d2h_done, cudaEventDisableTiming));
    }
    return DABGPU_OK;
}

}  // extern "C"

// The slot of the next ticket.  When the caller has not waited for the ticket that used it DABGPU_PIPELINE_DEPTH tickets ago,
// this waits for it: everything that ticket queued has then finished, its compute included.
static int pipe_acquire(dabgpu_ctx* ctx, dabgpu_ctx::PipeSlot** out) {
    int rc;
    if ((rc = pipe_init(ctx))) return rc;
    auto& sl = ctx->pipe[ctx->next_ticket % DABGPU_PIPELINE_DEPTH];
    if (sl.busy) { CUDA_TRY(cudaEventSynchronize(sl.d2h_done)); sl.busy = false; }
    *out = &sl;
    return DABGPU_OK;
}

// Everything of a ticket after its OFDM stage, which the caller has queued on the compute stream: the newest frame of every
// stream that produced one (during the last OFDM run, or since the counters in d_written0 when given), the channel decode,
// the DAB+ pack when dp is given (dp_log = its bound, checked by dp_check_out), and the device->host copies of the non-NULL
// result pointers of st and of dp on the copy-out stream.
static int pipe_finish(dabgpu_ctx* ctx, dabgpu_ctx::PipeSlot& sl, const dabgpu_step* st, const uint32_t* d_written0, const dabgpu_dabplus_out* dp,
                       size_t dp_log, uint64_t* ticket) {
    int rc;
    OfdmState& O = ctx->ofdm;
    const int n = st->n_streams, first = st->first_stream;
    const size_t fb = size_t(ctx->P.nb_frame_bits);
    if (st->frames_host || st->produced_host) {
        if ((rc = sl.d_stage.alloc(size_t(n) * fb))) return rc;
        if ((rc = sl.d_produced.alloc(size_t(n)))) return rc;
        rc = d_written0 ? ofdm_gather_since(O, first, n, d_written0, sl.d_stage.as<int8_t>(), sl.d_produced.as<uint8_t>(), ctx->stream)
                        : ofdm_gather_latest(O, first, n, sl.d_stage.as<int8_t>(), sl.d_produced.as<uint8_t>(), ctx->stream);
        if (rc) return rc;
    }
    if (st->run_chan_decode && (rc = dabgpu_chan_decode(ctx, first, n))) return rc;
    CUDA_TRY(join_dabplus(ctx));
    // The pack reads the decode's event queues and superframes on the compute stream, after the join.  Ticket t + 1's channel
    // decode, which overwrites them, forks from this stream after this point, so the output is this ticket's decode; nothing
    // else orders the two.  It writes the slot's own buffer, so the next compute need not wait for the copy-out.
    if (dp && (rc = dp_pack(ctx, first, n, dp_log, sl.d_dpout))) return rc;
    CUDA_TRY(cudaEventRecord(sl.compute_done, ctx->stream));
    // Copy out.  The next compute may overwrite the channel-decode arenas: it is made to wait for this copy.
    CUDA_TRY(cudaStreamWaitEvent(ctx->s_d2h, sl.compute_done, 0));
    const int nb_cifs = ctx->P.nb_cifs;
    if (st->frames_host) CUDA_TRY(cudaMemcpyAsync(st->frames_host, sl.d_stage.p, size_t(n) * fb, cudaMemcpyDeviceToHost, ctx->s_d2h));
    if (st->produced_host) CUDA_TRY(cudaMemcpyAsync(st->produced_host, sl.d_produced.p, size_t(n), cudaMemcpyDeviceToHost, ctx->s_d2h));
    bool arenas = false;
    if (st->msc_host) { arenas = true; CUDA_TRY(cudaMemcpyAsync(st->msc_host, ctx->d_msc_out.as<uint8_t>() + size_t(first) * nb_cifs * CIF_OUT_STRIDE, size_t(n) * nb_cifs * CIF_OUT_STRIDE, cudaMemcpyDeviceToHost, ctx->s_d2h)); }
    if (st->msc_valid_host) { arenas = true; CUDA_TRY(cudaMemcpyAsync(st->msc_valid_host, ctx->d_msc_valid.as<uint8_t>() + size_t(first) * nb_cifs * ctx->max_subs, size_t(n) * nb_cifs * ctx->max_subs, cudaMemcpyDeviceToHost, ctx->s_d2h)); }
    if (st->fic_host) { arenas = true; CUDA_TRY(cudaMemcpyAsync(st->fic_host, ctx->d_fic_out.as<uint8_t>() + size_t(first) * nb_cifs * FIC_GROUP_BYTES, size_t(n) * nb_cifs * FIC_GROUP_BYTES, cudaMemcpyDeviceToHost, ctx->s_d2h)); }
    if (st->fic_crc_host) { arenas = true; CUDA_TRY(cudaMemcpyAsync(st->fic_crc_host, ctx->d_fic_crc.as<uint8_t>() + size_t(first) * nb_cifs * 4, size_t(n) * nb_cifs * 4, cudaMemcpyDeviceToHost, ctx->s_d2h)); }
    if (st->chan_status_host) { arenas = true; CUDA_TRY(cudaMemcpyAsync(st->chan_status_host, ctx->d_status.as<int32_t>() + 2 * size_t(first), size_t(n) * 8, cudaMemcpyDeviceToHost, ctx->s_d2h)); }
    if (dp && (rc = dp_copy_out(ctx, n, dp_log, sl.d_dpout, dp, ctx->s_d2h))) return rc;
    CUDA_TRY(cudaEventRecord(sl.d2h_done, ctx->s_d2h));
    if (arenas) CUDA_TRY(cudaStreamWaitEvent(ctx->stream, sl.d2h_done, 0));
    sl.busy = true;
    sl.ticket = ctx->next_ticket;
    *ticket = ctx->next_ticket++;
    return DABGPU_OK;
}

extern "C" {

int dabgpu_submit(dabgpu_ctx* ctx, const dabgpu_step* st, uint64_t* ticket) { return dabgpu_submit_ex(ctx, st, nullptr, ticket); }

// DAB+ output of a ticket: asked for with the channel decode it packs, and refused before anything is queued.
static int dp_check_step(dabgpu_ctx* ctx, const dabgpu_step* st, const dabgpu_dabplus_out* dp, size_t* dp_log) {
    if (!dp) return DABGPU_OK;
    if (!st->run_chan_decode) return set_error(DABGPU_ERR_INVALID, "DAB+ output needs run_chan_decode");
    return dp_check_out(ctx, st->first_stream, st->n_streams, dp, dp_log);
}

int dabgpu_submit_ex(dabgpu_ctx* ctx, const dabgpu_step* st, const dabgpu_dabplus_out* dp, uint64_t* ticket) {
    if (!ctx || !st || !ticket) return set_error(DABGPU_ERR_INVALID, "null argument");
    int rc = check_stream_range(ctx, st->first_stream, st->n_streams);
    if (rc) return rc;
    if (!st->iq_host || st->n_samples <= 0 || st->n_streams == 0) return set_error(DABGPU_ERR_INVALID, "bad IQ buffer");
    size_t dp_log = 0;
    if ((rc = dp_check_step(ctx, st, dp, &dp_log))) return rc;
    OfdmState& O = ctx->ofdm;
    if (O.external_ring) return set_error(DABGPU_ERR_STATE, "a device input buffer is attached: use dabgpu_ofdm_advance");
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(join_if_many_frames(ctx, st->n_samples));
    const uint64_t t = ctx->next_ticket;
    auto& prev = ctx->pipe[(t + DABGPU_PIPELINE_DEPTH - 1) % DABGPU_PIPELINE_DEPTH];
    // the copy of this step overlaps the compute of the previous one: together they must fit the ring headroom
    const size_t prev_samples = ctx->pipe_recent_samples[(t + DABGPU_PIPELINE_DEPTH - 1) % DABGPU_PIPELINE_DEPTH];
    if (size_t(st->n_samples) + prev_samples > ofdm_ring_headroom(O))
        return set_error(DABGPU_ERR_INVALID, "n_samples %d (+%zu in flight) exceeds the IQ ring headroom %zu: raise ring_samples", st->n_samples,
                         prev_samples, ofdm_ring_headroom(O));
    dabgpu_ctx::PipeSlot* sl;
    if ((rc = pipe_acquire(ctx, &sl))) return rc;
    const int n = st->n_streams, first = st->first_stream;
    // (1) copy in; the ring region being overwritten was last read by the compute two tickets ago, which pipe_acquire covers
    if (prev.busy) CUDA_TRY(cudaStreamWaitEvent(ctx->s_h2d, prev.h2d_done, 0));
    if ((rc = ofdm_upload(O, st->iq_host, st->iq_stride_bytes, first, n, 0, size_t(st->n_samples), ctx->s_h2d))) return rc;
    CUDA_TRY(cudaEventRecord(sl->h2d_done, ctx->s_h2d));
    // (2) compute
    CUDA_TRY(cudaStreamWaitEvent(ctx->stream, sl->h2d_done, 0));
    const int bs = st->block_size > 0 ? st->block_size : st->n_samples;
    ctx->ofdm.demod_ctas_cap = ctx->dp_pending ? 3 : 0;   // a channel decode is running on its stream: share the SMs with it
    if ((rc = ofdm_run(O, first, n, st->n_samples, bs, ctx->stream))) return rc;
    // (3) channel decode and copy out
    if ((rc = pipe_finish(ctx, *sl, st, nullptr, dp, dp_log, ticket))) return rc;
    ctx->pipe_recent_samples[t % DABGPU_PIPELINE_DEPTH] = size_t(st->n_samples);
    return DABGPU_OK;
}

int dabgpu_wait(dabgpu_ctx* ctx, uint64_t ticket) {
    if (!ctx) return set_error(DABGPU_ERR_INVALID, "null context");
    if (ticket == 0 || ticket >= ctx->next_ticket) return set_error(DABGPU_ERR_INVALID, "unknown ticket %llu", (unsigned long long)ticket);
    auto& sl = ctx->pipe[ticket % DABGPU_PIPELINE_DEPTH];
    if (!sl.busy || sl.ticket != ticket) return DABGPU_OK;   // already retired
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(cudaEventSynchronize(sl.d2h_done));
    sl.busy = false;
    return DABGPU_OK;
}

int dabgpu_msc_get_layout(dabgpu_ctx* ctx, int stream, int sub_index, int* offset, int* bytes_per_cif) {
    int rc = check_stream_range(ctx, stream, 1);
    if (rc) return rc;
    const auto& hs = ctx->subs[size_t(stream)];
    if (sub_index < 0 || size_t(sub_index) >= hs.size() || !hs[size_t(sub_index)].active) return set_error(DABGPU_ERR_INVALID, "sub-channel index %d not configured", sub_index);
    if (offset) *offset = int(hs[size_t(sub_index)].out_offset);
    if (bytes_per_cif) *bytes_per_cif = int(hs[size_t(sub_index)].n_out_bytes);
    return DABGPU_OK;
}

// ---------------------------------------------------------------------------------------------
// Wideband front end (kernel in wideband.cuh)
// ---------------------------------------------------------------------------------------------
}  // extern "C"

struct dabgpu_wideband {
    dabgpu_ctx* ctx = nullptr;   // null once the context was destroyed
    int D = 1, fmt = 0, bps = 2, n_sources = 0, n_channels = 0;
    long long fs = 0;
    dabgpu_wideband_geometry geo{};   // block geometry (dabgpu_wideband_plan)
    bool mixed = false;               // k_wideband_mixed (fft_in not a power of two) instead of k_wideband<D>
    std::vector<int> radices;         // forward FFT passes of k_wideband_mixed
    DevBuf d_ring, d_H, d_twf, d_twi, d_dposf, d_dposi, d_chans, d_first;
    int ring_log2 = 0;
    size_t ring_cap = 0, out_cap = 0, headroom = 0;
    unsigned long long max_pass_blocks = 0;
    float2* d_out = nullptr;
    unsigned long long n_in = 0, blocks_done = 0, out_consumed = 0;   // input samples per source, blocks filtered, outputs handed to OFDM
    size_t max_submit = 0;            // samples per source a ticket may carry (dabgpu_wideband_reserve); 0: none
};

// Input ring size (log2) for tickets of up to max_submit samples per source.  The ring keeps the history of the next block
// (fft_in - step_in samples), the input held back until that block is complete (< step_in) and either one pass of
// max_pass_blocks blocks, or two tickets: the upload of ticket t + 1 then writes none of the samples the filter passes of
// ticket t still read.
static int wb_ring_log2(const dabgpu_wideband* w, size_t max_submit) {
    const size_t ov_in = size_t(w->geo.fft_in - w->geo.step_in), step_in = size_t(w->geo.step_in);
    const size_t need = std::max<size_t>(ov_in + (w->max_pass_blocks + 1) * step_in, ov_in + step_in - 1 + 2 * max_submit);
    int log2 = 0;
    while ((size_t(1) << log2) < need) log2++;
    return log2;
}

static void wb_detach(dabgpu_wideband* w) {
    DevBuf* bufs[] = {&w->d_ring, &w->d_H, &w->d_twf, &w->d_twi, &w->d_dposf, &w->d_dposi, &w->d_chans, &w->d_first};
    for (DevBuf* b : bufs) b->release();
    if (w->ctx) w->ctx->wb = nullptr;
    w->ctx = nullptr;
}

// Kaiser-windowed sinc low-pass, unit DC gain: scipy.signal.firwin(T, 856e3, window=('kaiser', kaiser_beta(70)), fs)
static void wb_design_taps(int T, long long fs, std::vector<double>& h) {
    const double c = 856e3 / (0.5 * double(fs)), beta = 0.1102 * (70.0 - 8.7), alpha = 0.5 * (T - 1);
    auto i0 = [](double x) {
        double sum = 1.0, term = 1.0;
        for (int k = 1; k < 200 && term > 1e-18 * sum; k++) { const double q = x / (2.0 * k); term *= q * q; sum += term; }
        return sum;
    };
    h.assign(size_t(T), 0.0);
    double sum = 0.0;
    for (int n = 0; n < T; n++) {
        const double m = n - alpha, r = m / alpha;
        const double sinc = (m == 0.0) ? 1.0 : sin(M_PI * c * m) / (M_PI * c * m);
        h[size_t(n)] = c * sinc * i0(beta * sqrt(std::max(0.0, 1.0 - r * r))) / i0(beta);
        sum += h[size_t(n)];
    }
    for (double& v : h) v /= sum;
}

// DIF pass radices: those of fft_cta<n> for a power of two (8, 8, ..., then 4 or 2), else 8s, then 4 or 2, then 3s, then 5s
// (fft_mixed_fwd)
static std::vector<int> wb_radices(int n) {
    std::vector<int> radices;
    int m = n;
    while (m % 8 == 0) { radices.push_back(8); m /= 8; }
    if (m % 4 == 0) { radices.push_back(4); m /= 4; }
    if (m % 2 == 0) { radices.push_back(2); m /= 2; }
    while (m % 3 == 0) { radices.push_back(3); m /= 3; }
    while (m % 5 == 0) { radices.push_back(5); m /= 5; }
    return radices;
}

// padded position of natural index k in the digit-reversed output of an in-place DIF FFT of n points with these pass radices
static void wb_dpos(int n, const std::vector<int>& radices, std::vector<uint16_t>& dpos) {
    dpos.resize(size_t(n));
    for (int k = 0; k < n; k++) {
        int a = 0, rem = n, kk = k;
        for (int R : radices) { const int d = kk % R; kk /= R; rem /= R; a += d * rem; }
        dpos[size_t(k)] = uint16_t(OFDM_PAD(a));
    }
}

// exp(-j 2 pi k / n), k < count
static void wb_roots(int n, int count, std::vector<float2>& tw) {
    tw.resize(size_t(count));
    for (int k = 0; k < count; k++) tw[size_t(k)] = make_float2(float(cos(-2.0 * M_PI * k / n)), float(sin(-2.0 * M_PI * k / n)));
}

// block geometry at fs (include/dabgpu.h): among the bin spacings 4, 2 and 1 kHz that divide fs and give an N_in <= 8192 with
// no prime factor above 5, the one with the fewest inverse-FFT operations per output sample
static bool wb_plan(long long fs, dabgpu_wideband_geometry& out) {
    if (fs < 2048000 || fs > 32768000) return false;
    bool found = false;
    double best = 0.0;
    for (const int bin : {4000, 2000, 1000}) {
        if (fs % bin) continue;
        const int n_in = int(fs / bin);
        int m = n_in;
        for (const int p : {2, 3, 5})
            while (m % p == 0) m /= p;
        if (n_in > WB_MIX_MAX_FFT || m != 1) continue;
        const int n_out = 2048000 / bin, T = int(2 * ((fs + 63999) / 64000) + 1);
        const int ov_out = int(((long long)(T - 1) * 2048000 + fs - 1) / fs);
        const long long g = 2048000 / std::gcd(fs, 2048000LL), l = g / std::gcd(g, 64LL) * 64;
        const int step_out = int((n_out - ov_out) / l * l);
        if (step_out <= 0) continue;
        const double cost = 5.0 * n_out * std::log2(double(n_out)) / step_out;
        if (found && cost >= best) continue;
        found = true;
        best = cost;
        out.bin_hz = bin; out.fft_in = n_in; out.fft_out = n_out; out.taps = T;
        out.step_out = step_out; out.step_in = int((long long)step_out * fs / 2048000);
    }
    return found;
}

// one entry per (D, format): W == nullptr sets the kernel's shared-memory attribute, otherwise launches nb blocks of every source
typedef int (*WbKernelFn)(const WbDev* W, unsigned long long block0, unsigned nb, int n_sources, cudaStream_t cs);
template <int D, int FMT> static int wb_kernel_t(const WbDev* W, unsigned long long block0, unsigned nb, int n_sources, cudaStream_t cs) {
    if (!W) {
        CUDA_TRY(cudaFuncSetAttribute(k_wideband<D, FMT>, cudaFuncAttributeMaxDynamicSharedMemorySize, WbCfg<D>::SMEM));
        return DABGPU_OK;
    }
    k_wideband<D, FMT><<<dim3(nb, unsigned(n_sources)), 64 * D, WbCfg<D>::SMEM, cs>>>(*W, block0);
    CUDA_TRY(cudaGetLastError());
    return DABGPU_OK;
}
#define WB_ROW(D) {wb_kernel_t<D, 0>, wb_kernel_t<D, 1>, wb_kernel_t<D, 2>, wb_kernel_t<D, 3>}
static const WbKernelFn kWbKernels[5][4] = {WB_ROW(1), WB_ROW(2), WB_ROW(4), WB_ROW(8), WB_ROW(16)};
#undef WB_ROW
static WbKernelFn wb_kernel(int D, int fmt) { return kWbKernels[__builtin_ctz(unsigned(D))][fmt]; }

// the same for k_wideband_mixed, one entry per (NOUT, format)
typedef int (*WbMixKernelFn)(const WbMixDev* W, unsigned long long block0, unsigned nb, int n_sources, cudaStream_t cs);
template <int NOUT, int FMT> static int wb_mix_kernel_t(const WbMixDev* W, unsigned long long block0, unsigned nb, int n_sources, cudaStream_t cs) {
    if (!W) {
        CUDA_TRY(cudaFuncSetAttribute(k_wideband_mixed<NOUT, FMT>, cudaFuncAttributeMaxDynamicSharedMemorySize, WbMixCfg<NOUT>::SMEM_MAX));
        return DABGPU_OK;
    }
    const int smem = (2 * OFDM_PAD(W->n_fft) + WbMixCfg<NOUT>::GROUP_FLOATS) * int(sizeof(float));
    k_wideband_mixed<NOUT, FMT><<<dim3(nb, unsigned(n_sources)), WB_MIX_THREADS, smem, cs>>>(*W, block0);
    CUDA_TRY(cudaGetLastError());
    return DABGPU_OK;
}
#define WB_MIX_ROW(NOUT) {wb_mix_kernel_t<NOUT, 0>, wb_mix_kernel_t<NOUT, 1>, wb_mix_kernel_t<NOUT, 2>, wb_mix_kernel_t<NOUT, 3>}
static const WbMixKernelFn kWbMixKernels[3][4] = {WB_MIX_ROW(512), WB_MIX_ROW(1024), WB_MIX_ROW(2048)};
#undef WB_MIX_ROW
static WbMixKernelFn wb_mix_kernel(int n_out, int fmt) { return kWbMixKernels[__builtin_ctz(unsigned(n_out / 512))][fmt]; }

static int wb_check_ctx(const dabgpu_ctx* ctx) {
    if (ctx->wb) return set_error(DABGPU_ERR_STATE, "a wideband front end is already open on this context");
    if (ctx->cfg.iq_format != DABGPU_IQ_C32) return set_error(DABGPU_ERR_INVALID, "the wideband front end writes c32: the context needs DABGPU_IQ_C32");
    return DABGPU_OK;
}
static int wb_open(dabgpu_ctx* ctx, const dabgpu_wideband_config* cfg, const dabgpu_wideband_geometry& geo, void* d_out,
                   size_t capacity, dabgpu_wideband** out);

extern "C" {

int dabgpu_wideband_plan(int sample_rate, dabgpu_wideband_geometry* g) {
    if (!g) return set_error(DABGPU_ERR_INVALID, "null argument");
    if (!wb_plan(sample_rate, *g))
        return set_error(DABGPU_ERR_INVALID, "sample rate %d Hz is not supported: it must lie in [2 048 000, 32 768 000] and be "
                         "N x 4000, 2000 or 1000 Hz with N <= 8192 and no prime factor of N above 5", sample_rate);
    return DABGPU_OK;
}

int dabgpu_wideband_open(dabgpu_ctx* ctx, const dabgpu_wideband_config* cfg, void* d_out, size_t capacity, dabgpu_wideband** out) {
    if (!ctx || !cfg || !d_out || !out) return set_error(DABGPU_ERR_INVALID, "null argument");
    *out = nullptr;
    if (int rc = wb_check_ctx(ctx)) return rc;
    const int D = cfg->sample_rate / 2048000;
    if (cfg->sample_rate <= 0 || cfg->sample_rate % 2048000 != 0 || (D != 1 && D != 2 && D != 4 && D != 8 && D != 16))
        return set_error(DABGPU_ERR_INVALID, "sample rate %d Hz is not 2.048 MHz x 1, 2, 4, 8 or 16", cfg->sample_rate);
    dabgpu_wideband_geometry geo;
    wb_plan(cfg->sample_rate, geo);
    return wb_open(ctx, cfg, geo, d_out, capacity, out);
}

int dabgpu_wideband_open_any_rate(dabgpu_ctx* ctx, const dabgpu_wideband_config* cfg, void* d_out, size_t capacity, dabgpu_wideband** out) {
    if (!ctx || !cfg || !d_out || !out) return set_error(DABGPU_ERR_INVALID, "null argument");
    *out = nullptr;
    if (int rc = wb_check_ctx(ctx)) return rc;
    dabgpu_wideband_geometry geo;
    if (int rc = dabgpu_wideband_plan(cfg->sample_rate, &geo)) return rc;
    return wb_open(ctx, cfg, geo, d_out, capacity, out);
}

}  // extern "C"

static int wb_open(dabgpu_ctx* ctx, const dabgpu_wideband_config* cfg, const dabgpu_wideband_geometry& geo, void* d_out,
                   size_t capacity, dabgpu_wideband** out) {
    if (cfg->format < DABGPU_WB_RAW_U8 || cfg->format > DABGPU_WB_RAW_F32L) return set_error(DABGPU_ERR_INVALID, "bad wideband format %d", cfg->format);
    if (cfg->n_sources < 1 || cfg->n_sources > 65535) return set_error(DABGPU_ERR_INVALID, "n_sources %d out of range", cfg->n_sources);
    if (cfg->n_channels < 1 || cfg->n_channels > ctx->cfg.max_streams)
        return set_error(DABGPU_ERR_INVALID, "n_channels %d: the context holds %d streams", cfg->n_channels, ctx->cfg.max_streams);
    if (!cfg->source || !cfg->offset_hz) return set_error(DABGPU_ERR_INVALID, "null channel table");
    const long long fs = cfg->sample_rate;
    for (int c = 0; c < cfg->n_channels; c++) {
        if (cfg->source[c] < 0 || cfg->source[c] >= cfg->n_sources) return set_error(DABGPU_ERR_INVALID, "channel %d: source %d out of range", c, cfg->source[c]);
        if (std::llabs((long long)cfg->offset_hz[c]) + 768000 > fs / 2)
            return set_error(DABGPU_ERR_INVALID, "channel %d: offset %d Hz puts the ensemble outside +-fs/2", c, cfg->offset_hz[c]);
    }
    const size_t min_cap = size_t(ctx->P.nb_frame_samples) + size_t(ctx->P.nb_null_period + ctx->P.nb_symbol_period) + 1024 + size_t(geo.step_out);
    if (!is_pow2(capacity) || capacity < min_cap || capacity > (size_t(1) << 30))
        return set_error(DABGPU_ERR_INVALID, "capacity %zu: must be a power of two in [%zu, 2^30]", capacity, min_cap);

    dabgpu_wideband* w = new dabgpu_wideband();
    w->D = int(fs / 2048000); w->fmt = cfg->format; w->fs = fs;
    w->geo = geo;
    w->mixed = !is_pow2(size_t(geo.fft_in));
    w->bps = (cfg->format == DABGPU_WB_RAW_F32L) ? 8 : (cfg->format == DABGPU_WB_RAW_S16L) ? 4 : 2;
    w->n_sources = cfg->n_sources; w->n_channels = cfg->n_channels;
    w->out_cap = capacity;
    w->headroom = ofdm_ring_headroom(ctx->P, capacity);
    w->max_pass_blocks = std::min<unsigned long long>(512, w->headroom / size_t(geo.step_out));
    w->d_out = static_cast<float2*>(d_out);
    w->ring_log2 = wb_ring_log2(w, 0);
    w->ring_cap = size_t(1) << w->ring_log2;

    // channels grouped by source, in channel order
    std::vector<WbChan> chans;
    std::vector<int> first(size_t(cfg->n_sources) + 1, 0);
    for (int s = 0; s < cfg->n_sources; s++) {
        first[size_t(s)] = int(chans.size());
        for (int c = 0; c < cfg->n_channels; c++) {
            if (cfg->source[c] != s) continue;
            const int f = cfg->offset_hz[c];
            const int half = geo.bin_hz / 2;
            const int bin = f >= 0 ? (f + half) / geo.bin_hz : -((half - f) / geo.bin_hz);   // round half away from zero
            chans.push_back(WbChan{bin, f - geo.bin_hz * bin, c, 0});
        }
    }
    first[size_t(cfg->n_sources)] = int(chans.size());

    const int N = geo.fft_in, NO = geo.fft_out;
    std::vector<double> h;
    wb_design_taps(geo.taps, fs, h);
    std::vector<float2> H(static_cast<size_t>(NO)), twf, twi;
    for (int i = 0; i < NO; i++) {
        const int u = i < NO / 2 ? i : i - NO;
        double re = 0.0, im = 0.0;
        for (size_t n = 0; n < h.size(); n++) {
            const long long k = ((long long)u * (long long)n) % N;
            re += h[n] * cos(-2.0 * M_PI * double(k) / N);
            im += h[n] * sin(-2.0 * M_PI * double(k) / N);
        }
        H[size_t(i)] = make_float2(float(re / N), float(im / N));
    }
    wb_roots(N, w->mixed ? N : N / 8, twf);
    wb_roots(NO, NO / 8, twi);
    w->radices = wb_radices(N);
    std::vector<uint16_t> dposf, dposi;
    wb_dpos(N, w->radices, dposf);
    wb_dpos(NO, wb_radices(NO), dposi);

    int rc = DABGPU_OK;
#define WB_TRY(expr) do { if ((rc = (expr))) { wb_detach(w); delete w; return rc; } } while (0)
    cudaError_t e = cudaSetDevice(ctx->cfg.device);
    if (e != cudaSuccess) { delete w; return set_error(DABGPU_ERR_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e)); }
    WB_TRY(w->d_ring.alloc(size_t(cfg->n_sources) * w->ring_cap * size_t(w->bps)));
    WB_TRY(w->d_H.alloc(H.size() * sizeof(float2)));
    WB_TRY(w->d_twf.alloc(twf.size() * sizeof(float2)));
    WB_TRY(w->d_twi.alloc(twi.size() * sizeof(float2)));
    WB_TRY(w->d_dposf.alloc(dposf.size() * 2));
    WB_TRY(w->d_dposi.alloc(dposi.size() * 2));
    WB_TRY(w->d_chans.alloc(chans.size() * sizeof(WbChan)));
    WB_TRY(w->d_first.alloc(first.size() * sizeof(int)));
    const std::pair<DevBuf*, std::pair<const void*, size_t>> up[] = {
        {&w->d_H, {H.data(), H.size() * sizeof(float2)}}, {&w->d_twf, {twf.data(), twf.size() * sizeof(float2)}},
        {&w->d_twi, {twi.data(), twi.size() * sizeof(float2)}}, {&w->d_dposf, {dposf.data(), dposf.size() * 2}},
        {&w->d_dposi, {dposi.data(), dposi.size() * 2}}, {&w->d_chans, {chans.data(), chans.size() * sizeof(WbChan)}},
        {&w->d_first, {first.data(), first.size() * sizeof(int)}}};
    for (const auto& u : up) {
        e = cudaMemcpy(u.first->p, u.second.first, u.second.second, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) { wb_detach(w); delete w; return set_error(DABGPU_ERR_CUDA, "cudaMemcpy: %s", cudaGetErrorString(e)); }
    }
    WB_TRY(w->mixed ? wb_mix_kernel(NO, w->fmt)(nullptr, 0, 0, 0, ctx->stream) : wb_kernel(w->D, w->fmt)(nullptr, 0, 0, 0, ctx->stream));
    WB_TRY(ofdm_attach(ctx->ofdm, d_out, capacity, capacity, ctx->stream));
#undef WB_TRY
    w->ctx = ctx;
    ctx->wb = w;
    *out = w;
    return DABGPU_OK;
}

// Validation and set-up shared by dabgpu_wideband_process and _submit for a call of n_samples per source: the Process() block
// size (*bs) and the output samples per channel the call yields (*new_out).
static int wb_begin(dabgpu_wideband* w, size_t n_samples, int block_size, size_t* bs, size_t* new_out) {
    dabgpu_ctx* ctx = w->ctx;
    const size_t blk_out = size_t(w->geo.step_out);
    *new_out = size_t((w->n_in + n_samples) / (unsigned long long)w->geo.step_in - w->blocks_done) * blk_out;
    *bs = block_size > 0 ? size_t(block_size) : std::max<size_t>(*new_out, 1);
    if (*bs + blk_out > w->headroom)
        return set_error(DABGPU_ERR_INVALID, "block_size %zu does not fit the output ring (%zu samples of headroom)", *bs, w->headroom);
    CUDA_TRY(cudaSetDevice(ctx->cfg.device));
    CUDA_TRY(join_if_many_frames(ctx, long(std::min<size_t>(*new_out, 1ul << 40))));
    ctx->ofdm.demod_ctas_cap = ctx->dp_pending ? 3 : 0;   // a channel decode is running on its stream: share the SMs with it
    return DABGPU_OK;
}

// Queues the copy of n samples of every source (source s at src + s * stride) into the ring at n_in on cs.
static int wb_upload(dabgpu_wideband* w, const uint8_t* src, size_t stride, size_t n, cudaStream_t cs) {
    for (size_t left = n, off = 0; left > 0;) {
        const size_t pos = size_t(w->n_in & (w->ring_cap - 1)), run = std::min(left, w->ring_cap - pos);
        const size_t bytes = run * size_t(w->bps);
        CUDA_TRY(cudaMemcpy2DAsync(w->d_ring.as<uint8_t>() + pos * size_t(w->bps), w->ring_cap * size_t(w->bps), src + off * size_t(w->bps),
                                   w->n_sources > 1 ? stride : bytes, bytes, size_t(w->n_sources), cudaMemcpyHostToDevice, cs));
        w->n_in += run; off += run; left -= run;
    }
    return DABGPU_OK;
}

// One pass on the compute stream over the input in the ring: the filter bank over its whole blocks, at most max_pass_blocks
// and never more than the OFDM stage's headroom ahead of what that consumed, then OFDM_Demod::Process over the new outputs in
// blocks of bs.  A partial block only at the end of the call: once input_done and every complete block is filtered (*last).
static int wb_pass(dabgpu_wideband* w, size_t bs, bool input_done, bool* last) {
    dabgpu_ctx* ctx = w->ctx;
    const unsigned long long blk_in = (unsigned long long)w->geo.step_in;
    const size_t blk_out = size_t(w->geo.step_out);
    WbDev W;
    W.ring = w->d_ring.as<uint8_t>(); W.ring_log2 = w->ring_log2; W.ring_mask = w->ring_cap - 1;
    W.out = w->d_out; W.out_cap = w->out_cap;
    W.H = w->d_H.as<float2>(); W.tw_fwd = w->d_twf.as<float2>(); W.tw_inv = w->d_twi.as<float2>();
    W.dpos_fwd = w->d_dposf.as<uint16_t>(); W.dpos_inv = w->d_dposi.as<uint16_t>();
    W.chans = w->d_chans.as<WbChan>(); W.chan_first = w->d_first.as<int>(); W.fs = w->fs;
    WbMixDev M;
    M.w = W; M.n_fft = w->geo.fft_in; M.step_in = w->geo.step_in; M.ov_in = w->geo.fft_in - w->geo.step_in; M.step_out = w->geo.step_out;
    M.n_pass = int(w->radices.size());
    for (int p = 0; p < WB_MIX_MAX_PASSES; p++) M.radix[p] = p < M.n_pass ? w->radices[size_t(p)] : 1;
    const size_t pending = size_t(w->blocks_done * blk_out - w->out_consumed);
    const unsigned long long nb = std::min({w->n_in / blk_in - w->blocks_done, w->max_pass_blocks, (unsigned long long)((w->headroom - pending) / blk_out)});
    if (nb) {
        int rc = w->mixed ? wb_mix_kernel(w->geo.fft_out, w->fmt)(&M, w->blocks_done, unsigned(nb), w->n_sources, ctx->stream)
                          : wb_kernel(w->D, w->fmt)(&W, w->blocks_done, unsigned(nb), w->n_sources, ctx->stream);
        if (rc) return rc;
        ctx->launches++;
        w->blocks_done += nb;
    }
    const size_t avail = size_t(w->blocks_done * blk_out - w->out_consumed);
    *last = input_done && w->n_in / blk_in == w->blocks_done;
    const size_t present = *last ? avail : (avail / bs) * bs;
    if (present) {
        int rc = ofdm_run(ctx->ofdm, 0, w->n_channels, int(present), int(bs), ctx->stream);
        if (rc) return rc;
        w->out_consumed += present;
    }
    return DABGPU_OK;
}

extern "C" {

int dabgpu_wideband_process(dabgpu_wideband* w, const void* iq_host, size_t stride, size_t n_samples, int block_size, size_t* n_out) {
    if (!w) return set_error(DABGPU_ERR_INVALID, "null wideband front end");
    if (n_out) *n_out = 0;
    dabgpu_ctx* ctx = w->ctx;
    if (!ctx) return set_error(DABGPU_ERR_STATE, "the context of this wideband front end was destroyed");
    if (!iq_host && n_samples) return set_error(DABGPU_ERR_INVALID, "null input");
    if (w->n_sources > 1 && stride < n_samples * size_t(w->bps)) return set_error(DABGPU_ERR_INVALID, "source stride %zu is shorter than a source", stride);
    size_t bs, new_out;
    int rc = wb_begin(w, n_samples, block_size, &bs, &new_out);
    if (rc) return rc;
    const uint8_t* src = static_cast<const uint8_t*>(iq_host);
    const unsigned long long hist = (unsigned long long)(w->geo.fft_in - w->geo.step_in);
    size_t done = 0;
    for (bool last = false; !last;) {
        // input: the ring keeps everything from the first sample the next block reads (its fft_in - step_in samples of history)
        const unsigned long long keep = w->blocks_done * (unsigned long long)w->geo.step_in >= hist ? w->blocks_done * w->geo.step_in - hist : 0;
        const size_t take = std::min<size_t>(n_samples - done, size_t(keep + w->ring_cap - w->n_in));
        if ((rc = wb_upload(w, src + done * size_t(w->bps), stride, take, ctx->stream))) return rc;
        done += take;
        if ((rc = wb_pass(w, bs, done == n_samples, &last))) return rc;
    }
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (n_out) *n_out = new_out;
    return DABGPU_OK;
}

int dabgpu_wideband_reserve(dabgpu_wideband* w, size_t max_submit_samples) {
    if (!w) return set_error(DABGPU_ERR_INVALID, "null wideband front end");
    if (!w->ctx) return set_error(DABGPU_ERR_STATE, "the context of this wideband front end was destroyed");
    if (w->n_in > 0) return set_error(DABGPU_ERR_STATE, "dabgpu_wideband_reserve must come before the first input");
    if (max_submit_samples < 1 || max_submit_samples > size_t(INT_MAX))
        return set_error(DABGPU_ERR_INVALID, "max_submit_samples %zu out of range [1, %d]", max_submit_samples, INT_MAX);
    CUDA_TRY(cudaSetDevice(w->ctx->cfg.device));
    const int log2 = wb_ring_log2(w, max_submit_samples);
    if (log2 != w->ring_log2) {
        // the ring holds no input yet: nothing to keep
        const size_t row = size_t(w->n_sources) * size_t(w->bps);
        w->d_ring.release();
        if (int rc = w->d_ring.alloc(row << log2)) {
            w->d_ring.alloc(row << w->ring_log2);   // leave the front end as it was
            return rc;
        }
        w->ring_log2 = log2;
        w->ring_cap = size_t(1) << log2;
    }
    w->max_submit = max_submit_samples;
    return DABGPU_OK;
}

// Pipelined dabgpu_wideband_process + dabgpu_chan_decode: (1) the upload on the copy stream, (2) the filter bank and OFDM
// passes, the newest frames and the channel decode on the compute stream, (3) the copy-out, as in dabgpu_submit (pipe_finish).
int dabgpu_wideband_submit(dabgpu_wideband* w, const dabgpu_step* st, uint64_t* ticket) { return dabgpu_wideband_submit_ex(w, st, nullptr, ticket); }

int dabgpu_wideband_submit_ex(dabgpu_wideband* w, const dabgpu_step* st, const dabgpu_dabplus_out* dp, uint64_t* ticket) {
    if (!w || !st || !ticket) return set_error(DABGPU_ERR_INVALID, "null argument");
    dabgpu_ctx* ctx = w->ctx;
    if (!ctx) return set_error(DABGPU_ERR_STATE, "the context of this wideband front end was destroyed");
    const int first = st->first_stream, n = st->n_streams;
    if (first < 0 || n < 1 || first > w->n_channels - n)
        return set_error(DABGPU_ERR_INVALID, "channel range [%d,%d) is empty or outside [0,%d)", first, first + n, w->n_channels);
    if (!st->iq_host || st->n_samples <= 0) return set_error(DABGPU_ERR_INVALID, "bad input buffer");
    const size_t n_samples = size_t(st->n_samples);
    if (n_samples > w->max_submit)
        return set_error(DABGPU_ERR_INVALID, "n_samples %zu exceeds the %zu samples per ticket set with dabgpu_wideband_reserve", n_samples, w->max_submit);
    if (w->n_sources > 1 && st->iq_stride_bytes < n_samples * size_t(w->bps))
        return set_error(DABGPU_ERR_INVALID, "source stride %zu is shorter than a source", st->iq_stride_bytes);
    size_t dp_log = 0;
    int rc = dp_check_step(ctx, st, dp, &dp_log);
    if (rc) return rc;
    size_t bs, new_out;
    rc = wb_begin(w, n_samples, st->block_size, &bs, &new_out);
    if (rc) return rc;
    dabgpu_ctx::PipeSlot* sl;
    if ((rc = pipe_acquire(ctx, &sl))) return rc;
    const bool gather = st->frames_host || st->produced_host;
    if (gather && (rc = sl->d_written0.alloc(size_t(n) * 4))) return rc;
    // (1) copy in.  Ticket t - 1 may still be filtering: the reserve keeps this ticket's samples clear of what it reads.  The
    // ticket before that used this slot; its compute must have read its samples before they are overwritten.
    CUDA_TRY(cudaStreamWaitEvent(ctx->s_h2d, sl->compute_done, 0));
    if ((rc = wb_upload(w, static_cast<const uint8_t*>(st->iq_host), st->iq_stride_bytes, n_samples, ctx->s_h2d))) return rc;
    CUDA_TRY(cudaEventRecord(sl->h2d_done, ctx->s_h2d));
    // (2) compute
    CUDA_TRY(cudaStreamWaitEvent(ctx->stream, sl->h2d_done, 0));
    if (gather)
        CUDA_TRY(cudaMemcpyAsync(sl->d_written0.p, ctx->d_frames_written.as<uint32_t>() + first, size_t(n) * 4, cudaMemcpyDeviceToDevice, ctx->stream));
    for (bool last = false; !last;)
        if ((rc = wb_pass(w, bs, true, &last))) return rc;
    // (3) channel decode and copy out
    return pipe_finish(ctx, *sl, st, sl->d_written0.as<uint32_t>(), dp, dp_log, ticket);
}

int dabgpu_wideband_close(dabgpu_wideband* w) {
    if (!w) return set_error(DABGPU_ERR_INVALID, "null wideband front end");
    if (w->ctx) {
        cudaSetDevice(w->ctx->cfg.device);
        sync_ctx(w->ctx);
        if (w->ctx->s_d2h) cudaStreamSynchronize(w->ctx->s_d2h);   // the copy-out of tickets still in flight
    }
    wb_detach(w);
    delete w;
    return DABGPU_OK;
}

}  // extern "C"
