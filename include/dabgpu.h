/* include/dabgpu.h -- C ABI of libdabgpu.so, the B200 (sm_100a) DAB receive path.
 *
 * This is the drop-in boundary behind the reference's C++ classes.  Every entry point lists the
 * reference interface it replaces (paths relative to /root/reference/vendor/DAB-Radio/src unless
 * noted).  The reference classes are one-object-per-stream and synchronous; the ABI is the same
 * contract batched over many independent streams ("stream" = one tuner / one ensemble).
 *
 * Conventions
 *   - every function returns DABGPU_OK (0) or a negative dabgpu_status; nothing throws;
 *     dabgpu_last_error() gives a thread-local message for the last failure.
 *   - all buffers are caller-allocated plain memory; "host" pointers may be pageable or pinned,
 *     "device" pointers must belong to the context's CUDA device.
 *   - soft bits are int8: +127 = logical 1, -127 = logical 0, 0 = punctured (viterbi_config.h:11-14).
 *   - there is NO CPU fallback: without a CUDA device dabgpu_ctx_create fails with DABGPU_ERR_CUDA.
 */
#ifndef DABGPU_H
#define DABGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DABGPU_API __attribute__((visibility("default")))

typedef enum {
    DABGPU_OK = 0,
    DABGPU_ERR_INVALID = -1,   /* bad argument (e.g. invalid transmission mode: dab_ofdm_params_ref.cpp:53-54) */
    DABGPU_ERR_CUDA = -2,      /* CUDA runtime/driver failure or no device */
    DABGPU_ERR_NOMEM = -3,
    DABGPU_ERR_STATE = -4,     /* call not valid in the current state (e.g. nothing configured) */
    DABGPU_ERR_OVERFLOW = -5   /* caller buffer or internal queue too small */
} dabgpu_status;

typedef struct dabgpu_ctx dabgpu_ctx;

/* ---------------------------------------------------------------------------------------------
 * Context
 * ------------------------------------------------------------------------------------------- */
enum { DABGPU_IQ_U8 = 0, DABGPU_IQ_C32 = 1 };

/* Synchronisation knobs = OFDM_Demod_Config (ofdm/ofdm_demodulator.h:24-45), same defaults. */
typedef struct {
    float signal_l1_update_beta;      /* 0.95 */
    int   signal_l1_nb_samples;       /* 100  */
    int   signal_l1_nb_decimate;      /* 5    */
    float null_thresh_start;          /* 0.35 */
    float null_thresh_end;            /* 0.75 */
    float fine_freq_update_beta;      /* 0.9  */
    int   is_coarse_freq_correction;  /* 1    */
    float max_coarse_freq_correction_norm; /* 0.5 */
    float coarse_freq_slow_beta;      /* 0.1  */
    float impulse_peak_threshold_db;  /* 20   */
    float impulse_peak_distance_probability; /* 0.15 */
} dabgpu_ofdm_config;

typedef struct {
    int device;            /* CUDA device ordinal */
    int transmission_mode; /* 1..4 (get_DAB_OFDM_params / get_dab_parameters) */
    int max_streams;       /* independent IQ streams held by this context */
    int iq_format;         /* DABGPU_IQ_U8 (2 B/sample, converted on device like app_iq_readers.h:23-43,72-87) or DABGPU_IQ_C32 */
    size_t ring_samples;   /* per-stream IQ ring capacity in samples, power of two; 0 = 4 frames rounded up */
    int frame_slots;       /* soft-bit frame ring depth per stream, power of two >= the 16-CIF de-interleaver history + 2 frames
                              (8 in mode I, 16 in mode IV, 32 in modes II/III); 0 = twice that minimum */
    int max_subchannels;   /* sub-channel table size per stream; 0 = 64 */
    void* cuda_stream;     /* optional cudaStream_t owned by the caller; NULL = library creates one */
    dabgpu_ofdm_config ofdm;
    unsigned flags;        /* DABGPU_FLAG_* */
} dabgpu_config;
#define DABGPU_FLAG_NO_FIC 1u   /* dabgpu_chan_decode skips the FIC (contexts that only serve MSC_Decoder::DecodeCIF) */
/* Viterbi mapping.  Default: calls with thousands of trellises run one trellis per lane (k_viterbi_lanes), smaller calls
 * one trellis per warp (k_viterbi); both are bit-exact with the reference.  These flags pin one mapping (tests, profiling). */
#define DABGPU_FLAG_VIT_LANES_ALWAYS 2u
#define DABGPU_FLAG_VIT_LANES_NEVER 4u
/* Keep the synchronisation responses of every stream on the device for the GUI taps (dabgpu_ofdm_get_response). */
#define DABGPU_FLAG_DIAG_TAPS 8u

DABGPU_API const char* dabgpu_version(void);
DABGPU_API const char* dabgpu_last_error(void);
DABGPU_API int dabgpu_device_count(void);
DABGPU_API void dabgpu_config_default(dabgpu_config* cfg, int transmission_mode);
DABGPU_API int dabgpu_ctx_create(const dabgpu_config* cfg, dabgpu_ctx** out);
DABGPU_API void dabgpu_ctx_destroy(dabgpu_ctx* ctx);
DABGPU_API int dabgpu_sync(dabgpu_ctx* ctx);                       /* wait for all queued work */
/* Page-locked host memory for the buffers handed to dabgpu_submit / dabgpu_ofdm_process (copies from pageable memory neither
 * overlap nor reach the link rate).  write_combined != 0: for input buffers the CPU only ever writes.  Allocate on a thread
 * that is bound to the NUMA node of the GPU: the pages are placed where the calling thread runs. */
DABGPU_API int dabgpu_host_alloc(void** out, size_t bytes, int write_combined);
DABGPU_API void dabgpu_host_free(void* p);
DABGPU_API void* dabgpu_cuda_stream(dabgpu_ctx* ctx);              /* the stream every kernel is launched on */
/* number of kernels of this library launched on the context so far (bench.py "gpu_launches") */
DABGPU_API uint64_t dabgpu_launch_count(const dabgpu_ctx* ctx);

/* Device-side timing of the library's kernels by class (CUDA events on the launching stream), for roofline
 * reports.  The analogue of the reference's in-process profiler (ofdm/profiler.h).  Disabled by default. */
enum { DABGPU_PROF_OFDM_CTL = 0, DABGPU_PROF_OFDM_DEMOD = 1, DABGPU_PROF_VITERBI = 2, DABGPU_PROF_DABPLUS = 3,
       DABGPU_PROF_CHAN_MISC = 4, DABGPU_PROF_CLASSES = 5 };
typedef struct { double ms[DABGPU_PROF_CLASSES]; uint64_t launches[DABGPU_PROF_CLASSES]; } dabgpu_profile;
DABGPU_API int dabgpu_profile_enable(dabgpu_ctx* ctx, int on);   /* also clears the accumulated totals */
DABGPU_API int dabgpu_profile_read(dabgpu_ctx* ctx, dabgpu_profile* out);

/* Frame geometry: OFDM_Params (ofdm/ofdm_params.h) + DAB_Parameters (dab/constants/dab_parameters.h:5-24) */
typedef struct {
    int nb_frame_symbols, nb_symbol_period, nb_null_period, nb_cyclic_prefix, nb_fft, nb_data_carriers;
    int nb_frame_bits, nb_fic_bits, nb_msc_bits, nb_cifs, nb_fibs_per_cif, nb_fib_group_bits, nb_cif_bits;
    int nb_frame_samples;
} dabgpu_params;
DABGPU_API int dabgpu_get_params(int transmission_mode, dabgpu_params* out);

/* ---------------------------------------------------------------------------------------------
 * OFDM demodulation.  Replaces OFDM_Demod::{Process,Reset,On_OFDM_Frame,Get*}
 * (ofdm/ofdm_demodulator.h:109-141, ofdm_demodulator.cpp:235-950) with the canonical
 * serialised ordering of SURVEY.md appendix C: a completed frame is fully demodulated (and the
 * fine frequency updated) before the next sample of that stream is consumed.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    int state;                 /* OFDM_Demod::State numbering (ofdm_demodulator.h:50-56) */
    int total_frames_read;
    int total_frames_desync;
    int fine_time_offset;
    float signal_l1_average;
    float freq_coarse_offset;
    float freq_fine_offset;
    int frames_queued;         /* soft-bit frames produced and not yet popped */
    int frames_dropped;        /* frames dabgpu_ofdm_pop_frames could not deliver because the caller fell more than frame_slots-1
                                  frames behind and the ring slots were reused (the reference's observers never lose a frame) */
} dabgpu_ofdm_status;

/* OFDM_Demod::GetConfig() is mutable in the reference (the GUI edits it while running, ofdm_demodulator.h:122):
 * replaces the synchronisation knobs of every stream of the context from the next process/advance call on. */
DABGPU_API int dabgpu_ofdm_set_config(dabgpu_ctx* ctx, const dabgpu_ofdm_config* cfg);

/* OFDM_Demod::Reset() for one stream (-1 = all streams) */
DABGPU_API int dabgpu_ofdm_reset(dabgpu_ctx* ctx, int stream);

/* OFDM_Demod::Process(block) for streams [first_stream, first_stream+n_streams): copies n_samples
 * per stream from host memory (stream i at iq_host + i*stream_stride_bytes) into the device IQ
 * rings and consumes them.  The samples are presented to the state machine as consecutive
 * Process() calls of block_size samples (the reference's results depend on that partition while
 * acquiring, SURVEY.md H3; the CLI default is 65536).  block_size <= 0 means one block. */
DABGPU_API int dabgpu_ofdm_process(dabgpu_ctx* ctx, const void* iq_host, size_t stream_stride_bytes,
                                   int first_stream, int n_streams, int n_samples, int block_size);

/* Same, for IQ already resident in device memory (no copy): the caller's buffer replaces the
 * internal rings.  Layout: stream i sample k at d_iq + (i*stream_stride_samples + (k mod capacity))
 * * bytes_per_sample, k = absolute sample index since attach.  capacity must be a power of two or
 * >= every absolute index ever consumed. */
DABGPU_API int dabgpu_ofdm_attach_device_input(dabgpu_ctx* ctx, const void* d_iq, size_t stream_stride_samples,
                                               size_t capacity_samples);
DABGPU_API int dabgpu_ofdm_advance(dabgpu_ctx* ctx, int first_stream, int n_streams, int n_samples, int block_size);

/* ---------------------------------------------------------------------------------------------
 * Wideband front end.  Replaces, for every ensemble of a multi-ensemble capture at once, the 2.048 MHz VFO that
 * DABModule::enable puts in front of OFDM_Demod in the plugin (SURVEY.md 3.1) and the reference's
 * examples/apply_frequency_shift (SURVEY.md 2.1): mix each ensemble to baseband, low-pass filter and decimate to 2.048 MS/s.
 *
 * A source is one capture at fs = D x 2 048 000 Hz, D in {1, 2, 4, 8, 16}, in one of the formats below, scaled exactly as
 * dabgpu_iq_convert scales it.  Channel c (= context stream c) is the ensemble of source[c] centred offset_hz[c] above the
 * capture centre, |offset_hz[c]| + 768 000 <= fs / 2.  With h = firwin(64 D + 1, 856 kHz, Kaiser beta = kaiser_beta(70 dB))
 * (unit DC gain, computed in double on the host), f^ = 4000 round(f / 4000) (half away from zero), delta = f - f^, input before
 * sample 0 = 0, output n of a channel is
 *     y[n] = exp(-j 2 pi delta n D / fs) * sum_{i=0}^{64 D} h[i] x[n D - i] exp(-j 2 pi f^ (n D - i) / fs)
 * up to the aliasing beyond 1.024 MHz that the frequency-domain decimation drops (>= 75 dB down).  Every phase comes from the
 * absolute sample index in exact integer arithmetic modulo fs, so nothing drifts.  After n_in input samples per source, every
 * channel holds 448 floor(n_in / (448 D)) output samples; output n depends only on the input and n, whatever the call sizes.
 *
 * dabgpu_wideband_open_any_rate accepts every integer fs that dabgpu_wideband_plan supports (2.048 to 32.768 MS/s, e.g. the
 * 2.4, 2.5, 3, 6, 8, 10, 12.5 and 20 MS/s of common tuners) under the same offset rule.  With the plan's bin spacing Delta, T
 * taps h = firwin(T, 856 kHz, same Kaiser window, unit DC gain) at fs, f^ = Delta round(f / Delta) (half away from zero),
 * delta = f - f^ and input before sample 0 = 0, let
 *     v[m] = sum_{i<T} h[i] x[m - i] exp(-j 2 pi f^ (m - i) / fs).
 * Output n is exp(-j 2 pi delta n / 2 048 000) times the band-limited (|f| < 1.024 MHz) interpolation of v evaluated at input
 * time n fs / 2 048 000, up to the same >= 75 dB aliasing; where n fs / 2 048 000 is an integer this is the formula above.  All
 * phases are exact integers modulo N_in and 2 048 000.  After n_in input samples per source every channel holds
 * step_out floor(n_in / step_in) output samples, whatever the call sizes.  At fs = 2.048 MHz x 2^d the output is bit-identical
 * to dabgpu_wideband_open's.
 * ------------------------------------------------------------------------------------------- */
enum { DABGPU_WB_RAW_U8 = 0, DABGPU_WB_RAW_S8 = 1, DABGPU_WB_RAW_S16L = 2, DABGPU_WB_RAW_F32L = 3 };   /* the reference's mode strings */
typedef struct {
    int sample_rate;        /* Hz, 2 048 000 x {1, 2, 4, 8, 16}, shared by every source */
    int format;             /* DABGPU_WB_*, shared by every source */
    int n_sources;
    int n_channels;         /* <= max_streams of the context */
    const int* source;      /* [n_channels] source of channel c */
    const int* offset_hz;   /* [n_channels] centre of channel c relative to the capture centre, Hz */
} dabgpu_wideband_config;
typedef struct dabgpu_wideband dabgpu_wideband;
/* Block geometry of the filter bank at one rate.  bin_hz = Delta in {4000, 2000, 1000}; fft_in = fs / Delta (<= 8192, no prime
 * factor above 5) forward-FFT points per block; fft_out = 2 048 000 / Delta inverse-FFT points per channel; each block advances
 * step_in input and step_out output samples (step_in / step_out = fs / 2 048 000); taps = T = 2 ceil(fs / 64 000) + 1.  Of
 * the Delta that qualify, the plan takes the one with the fewest inverse-FFT operations per output sample.  At
 * 2.048 MHz x D: Delta = 4000, fft_in = 512 D, steps 448 D / 448, T = 64 D + 1. */
typedef struct {
    int bin_hz, fft_in, fft_out, step_in, step_out, taps;
} dabgpu_wideband_geometry;
/* Fills *g for sample_rate, or returns DABGPU_ERR_INVALID (with a message) when the rate is not supported.  Needs no device. */
DABGPU_API int dabgpu_wideband_plan(int sample_rate, dabgpu_wideband_geometry* g);
/* Validates cfg and attaches d_out (c32, channel c sample k at d_out[c * capacity_samples + (k mod capacity_samples)], the layout
 * of dabgpu_ofdm_attach_device_input with stride = capacity) to the context: every stream is reset, and dabgpu_ofdm_process /
 * dabgpu_submit return DABGPU_ERR_STATE from then on.  capacity_samples: power of two that holds a transmission frame, the
 * NULL + PRS window and a margin of 1472 samples.  The context must be created with DABGPU_IQ_C32; one front end per context
 * (a second open returns DABGPU_ERR_STATE).  Close it before destroying the context. */
DABGPU_API int dabgpu_wideband_open(dabgpu_ctx* ctx, const dabgpu_wideband_config* cfg, void* d_out, size_t capacity_samples,
                                    dabgpu_wideband** out);
/* dabgpu_wideband_open for any rate dabgpu_wideband_plan supports (cfg->sample_rate); capacity_samples must hold a transmission
 * frame, the NULL + PRS window and a margin of 1024 + step_out samples.  Process and close as for dabgpu_wideband_open. */
DABGPU_API int dabgpu_wideband_open_any_rate(dabgpu_ctx* ctx, const dabgpu_wideband_config* cfg, void* d_out,
                                             size_t capacity_samples, dabgpu_wideband** out);
/* Copies n_samples raw samples of every source (source s at iq_host + s * source_stride_bytes) to the device, filters them into
 * d_out and runs OFDM_Demod::Process on channels [0, n_channels) over the new output samples, presented as Process() blocks of
 * block_size (<= 0: one block).  Returns once the host buffer may be reused; *n_out = output samples per channel this call. */
DABGPU_API int dabgpu_wideband_process(dabgpu_wideband* w, const void* iq_host, size_t source_stride_bytes, size_t n_samples,
                                       int block_size, size_t* n_out);
/* Closes the front end once every queued call and the copy-out of every ticket in flight have finished. */
DABGPU_API int dabgpu_wideband_close(dabgpu_wideband* w);

/* On_OFDM_Frame: number of undelivered soft-bit frames per stream, then copy them out in order.
 * Each frame is nb_frame_bits int8.  infos (optional) receives per-frame {coarse, fine} offsets
 * and fine time offset as observed when the frame was emitted. */
typedef struct { float freq_coarse_offset, freq_fine_offset; int fine_time_offset; int frame_index; } dabgpu_frame_info;
DABGPU_API int dabgpu_ofdm_get_status(dabgpu_ctx* ctx, int stream, dabgpu_ofdm_status* out);
/* GUI taps served from device buffers (contexts created with DABGPU_FLAG_DIAG_TAPS): nb_fft floats in dB of the last
 * synchronisation of the stream.  kind 0 = OFDM_Demod::GetImpulseResponse (fine time correlation, ofdm_demodulator.cpp:473-548),
 * kind 1 = OFDM_Demod::GetCoarseFrequencyResponse (ofdm_demodulator.cpp:360-471), both read by the plugin's render code
 * (src/render_radio_block.cpp:192-214). */
DABGPU_API int dabgpu_ofdm_get_response(dabgpu_ctx* ctx, int stream, int kind, float* out, int n_floats);
/* OFDM_Demod::GetCorrelationTimeBuffer (ofdm_demodulator.h:139): the (nb_null_period + nb_symbol_period) complex<float> samples
 * of the NULL symbol + PRS window the synchronisation works on (no flag needed: the control kernel keeps it anyway). */
DABGPU_API int dabgpu_ofdm_get_correlation_buffer(dabgpu_ctx* ctx, int stream, float* out, size_t n_floats);
/* OFDM_Demod::GetFrameFFT (ofdm_demodulator.h:135): nb_frame_symbols x nb_fft complex<float> spectra (PRS first, natural bin
 * order) of the last frame the stream emitted, recomputed on demand from the IQ still in the device ring.  When n_floats has
 * room for (nb_frame_symbols + 1) rows, the last row is the spectrum of the NULL symbol that follows the frame, as in the
 * reference's buffer (ofdm_demodulator.cpp:108, 703-709).  DABGPU_ERR_STATE until a frame that lies contiguously in the ring has
 * been emitted. */
DABGPU_API int dabgpu_ofdm_get_frame_fft(dabgpu_ctx* ctx, int stream, float* out, size_t n_floats);
/* OFDM_Demod::GetFrameDataVec (ofdm_demodulator.h:136, CalculateDQPSK ofdm_demodulator.cpp:842-865): (nb_frame_symbols - 1) x
 * nb_data_carriers complex<float> differential vectors X_i * conj(X_{i+1}) of the same frame, carriers -K/2..K/2 without DC,
 * before the frequency de-interleaver (the constellation the GUI plots). */
DABGPU_API int dabgpu_ofdm_get_frame_data_vec(dabgpu_ctx* ctx, int stream, float* out, size_t n_floats);
DABGPU_API int dabgpu_ofdm_pop_frames(dabgpu_ctx* ctx, int stream, int8_t* frames_host, int max_frames,
                                      dabgpu_frame_info* infos, int* n_frames_out);
/* Bulk variant used by throughput harnesses: newest frame of every stream in [first, first+n) that
 * produced one during the last process/advance call is copied to frames_host + i*nb_frame_bits;
 * produced[i] = 1/0. */
DABGPU_API int dabgpu_ofdm_fetch_latest(dabgpu_ctx* ctx, int first_stream, int n_streams, int8_t* frames_host,
                                        uint8_t* produced);

/* Pipelined variant for throughput hosts (SURVEY.md section 7 "hard part 5": pinned, double-buffered staging).
 * dabgpu_submit queues, without blocking, (1) the host->device copy of n_samples per stream on a copy stream,
 * (2) the OFDM kernels and, if run_chan_decode != 0, the channel decode of the frames they produce on the compute
 * stream, (3) the device->host copy of whatever result pointers are non-NULL on a third stream.  dabgpu_wait blocks
 * until the results of that ticket are in host memory.  At most DABGPU_PIPELINE_DEPTH tickets are in flight: submit
 * waits for the oldest one when the pipeline is full.  Host buffers should be pinned (cudaHostAlloc / cudaHostRegister)
 * for the copies to overlap; they must stay valid until the ticket was waited for.  The reference analogue is the
 * reader thread / pipeline thread split of OFDM_Demod (ofdm/ofdm_demodulator_threads.h) plus the ThreadedRingBuffer
 * between OFDM_Demod and BasicRadio (src/radio_block.cpp:20-44). */
#define DABGPU_PIPELINE_DEPTH 2
#define DABGPU_CIF_OUT_STRIDE 6912   /* decoded bytes of one CIF never exceed 55296/8 */
#define DABGPU_FIC_GROUP_STRIDE 128
typedef struct {
    const void* iq_host;        /* stream i at iq_host + i*iq_stride_bytes */
    size_t iq_stride_bytes;
    int first_stream, n_streams, n_samples, block_size;
    int run_chan_decode;
    /* optional outputs (NULL = not copied) */
    int8_t* frames_host;        /* [n_streams][nb_frame_bits] newest soft-bit frame of each stream */
    uint8_t* produced_host;     /* [n_streams] 1 if the stream produced a frame in this step */
    uint8_t* msc_host;          /* [n_streams][nb_cifs][DABGPU_CIF_OUT_STRIDE] decoded sub-channel bytes (offsets: dabgpu_msc_get_layout) */
    uint8_t* msc_valid_host;    /* [n_streams][nb_cifs][max_subchannels] */
    uint8_t* fic_host;          /* [n_streams][nb_cifs][DABGPU_FIC_GROUP_STRIDE] */
    uint8_t* fic_crc_host;      /* [n_streams][nb_cifs][4] */
    int32_t* chan_status_host;  /* [n_streams][2] = {decoded, frame_index} */
} dabgpu_step;
DABGPU_API int dabgpu_submit(dabgpu_ctx* ctx, const dabgpu_step* step, uint64_t* ticket);
DABGPU_API int dabgpu_wait(dabgpu_ctx* ctx, uint64_t ticket);
/* byte offset and length of sub-channel sub_index inside one CIF row of the msc_host arena */
DABGPU_API int dabgpu_msc_get_layout(dabgpu_ctx* ctx, int stream, int sub_index, int* offset, int* bytes_per_cif);

/* Pipelined wideband front end (dabgpu_wideband_open above, the pipeline of dabgpu_submit).
 *
 * dabgpu_wideband_reserve sizes the device input ring for tickets of up to max_submit_samples raw samples per source: it holds
 * the fft_in - step_in samples of history of the next block, fewer than step_in samples held back until that block is
 * complete, and two tickets, rounded up to a power of two (one 96 ms frame per ticket at 16.384 MS/s raw_s16l for 128 sources
 * is about 2 GB).  Valid only before the first input (dabgpu_wideband_process or _submit), DABGPU_ERR_STATE after it; a failed
 * allocation is reported here (DABGPU_ERR_NOMEM) and leaves the front end as it was.  Outputs do not depend on the ring size.
 *
 * dabgpu_wideband_submit queues one ticket without blocking: (1) the copy of step->n_samples (1 .. the reserved size) raw
 * samples of every source (source s at step->iq_host + s * step->iq_stride_bytes) into the ring on the copy stream, (2) the
 * filter bank and OFDM_Demod::Process over every channel as dabgpu_wideband_process runs them (Process() blocks of
 * step->block_size), then, if step->run_chan_decode != 0, one dabgpu_chan_decode of channels [first_stream, first_stream +
 * n_streams) on the compute stream, (3) the copy of the non-NULL result pointers of step on the copy-out stream, in the layouts
 * of dabgpu_submit with row 0 = channel first_stream.  Tickets retire with dabgpu_wait and share the context's
 * DABGPU_PIPELINE_DEPTH slots.  Contract: after the same sequence of n_samples and block_size, ticket i leaves the device
 * state and the copied arenas exactly as dabgpu_wideband_process(n_i) followed by dabgpu_chan_decode(first, n) would.
 * produced_host[c] is 1 when channel first_stream + c emitted at least one frame during this ticket (which can span several
 * OFDM runs), and frames_host row c then holds the newest such frame.
 *
 * Ordering: the input must stay valid until the ticket was waited for and be pinned (dabgpu_host_alloc) for the copies to
 * overlap.  The upload of ticket t + 1 overlaps the compute of ticket t; the upload of ticket t + 2 waits for the compute of
 * ticket t.  dabgpu_wideband_process and _submit may be mixed in any order: each call's work is ordered after the previous
 * one's.  dabgpu_submit keeps returning DABGPU_ERR_STATE while a front end is attached. */
DABGPU_API int dabgpu_wideband_reserve(dabgpu_wideband* w, size_t max_submit_samples);
DABGPU_API int dabgpu_wideband_submit(dabgpu_wideband* w, const dabgpu_step* step, uint64_t* ticket);

/* ---------------------------------------------------------------------------------------------
 * Viterbi.  Replaces DAB_Viterbi_Decoder::{reset,update,chainback}
 * (dab/algorithms/dab_viterbi_decoder.h:22-33; decoder selected at dab_viterbi_decoder.cpp:51-73 =
 * ViterbiDecoder_AVX_u16<7,4>: saturating u16 metrics, tie => decision 1, renormalise at 60455).
 * One job = reset(); update(seg 0..n_seg-1); chainback(n_out_bytes).
 * ------------------------------------------------------------------------------------------- */
#define DABGPU_MAX_SEGMENTS 5
typedef struct {
    uint64_t soft_offset;       /* offset of the first punctured symbol inside the soft buffer */
    uint32_t n_soft;            /* punctured symbols available to this job */
    uint32_t n_seg;
    uint8_t  seg_pi[DABGPU_MAX_SEGMENTS + 3];   /* 1..24 = PI_TABLE row (puncture_codes.h:42-67), 0 = PI_X tail code */
    uint32_t seg_bits[DABGPU_MAX_SEGMENTS];     /* requested_output_symbols of each update() call (multiple of 4) */
    uint64_t out_offset;        /* byte offset inside the output buffer */
    uint32_t n_out_bytes;       /* chainback length in bytes */
    uint32_t descramble;        /* != 0: XOR with the energy-dispersal PRBS (additive_scrambler.h:10-36) */
} dabgpu_viterbi_job;

/* soft_host/out_host/path_error_host are host buffers; path_error_host (optional) gets the value
 * chainback() returns (accumulated renormalisation bias + final state-0 metric). */
DABGPU_API int dabgpu_viterbi_decode(dabgpu_ctx* ctx, const dabgpu_viterbi_job* jobs, int n_jobs,
                                     const int8_t* soft_host, size_t soft_bytes,
                                     uint8_t* out_host, size_t out_bytes, uint64_t* path_error_host);

/* FIC_Decoder::DecodeFIBGroup (dab/fic/fic_decoder.cpp:53-117) for n_groups independent FIB groups of 2304 soft
 * bits each (PI_16 x 21, PI_15 x 3, tail; energy dispersal; CRC16 per FIB).  fibs_host receives n_groups x 3 x 32
 * descrambled bytes (30 data + 2 CRC), crc_ok one flag per FIB. */
DABGPU_API int dabgpu_fic_decode(dabgpu_ctx* ctx, const int8_t* soft_host, int n_groups, uint8_t* fibs_host, uint8_t* crc_ok);

/* ---------------------------------------------------------------------------------------------
 * Channel decode of whole transmission frames.
 *   FIC  : replaces BasicFICRunner::Process + FIC_Decoder::DecodeFIBGroup (dab/fic/fic_decoder.cpp:53-117)
 *   MSC  : replaces MSC_Decoder::DecodeCIF = CIF_Deinterleaver + EEP/UEP depuncture + Viterbi + descramble
 *          (dab/msc/msc_decoder.cpp:46-154, dab/msc/cif_deinterleaver.cpp:20-71)
 *   DAB+ : replaces AAC_Frame_Processor::Process through RS(120,110), fire code and AU CRC
 *          (dab/audio/aac_frame_processor.cpp:126-362, dab/algorithms/reed_solomon_decoder.cpp:192-477)
 * Frames are taken from the per-stream soft-bit frame ring, which is filled either by the OFDM
 * stage on the device or by dabgpu_softbits_push (the BasicRadio::Process(span<viterbi_bit_t>) seam,
 * basic_radio/basic_radio.cpp:41-65).
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    int start_address;   /* in capacity units (64 soft bits) */
    int length;          /* in capacity units */
    int is_uep;
    int uep_prot_index;  /* UEP_PROTECTION_TABLE row (subchannel_protection_tables.h:21-86) */
    int eep_prot_level;  /* 0..3 = level 1..4 */
    int eep_type_b;      /* 0 = EEP-A, 1 = EEP-B */
    int is_dabplus;      /* run the DAB+ superframe stage on this sub-channel */
} dabgpu_subchannel;

/* Declares the MSC_Decoder set of one stream.  Entries that are identical to the entry with the same index of the previous
 * table keep their time de-interleaver and superframe state (BasicRadio never disturbs a running decoder, basic_radio.cpp:98-131);
 * every other entry starts empty like a new MSC_Decoder / AAC_Frame_Processor. */
DABGPU_API int dabgpu_msc_configure(dabgpu_ctx* ctx, int stream, const dabgpu_subchannel* subs, int n_subs);
/* BasicRadio::UpdateAfterProcessing (basic_radio/basic_radio.cpp:83-154): attach a decoder to one newly complete sub-channel;
 * the decoders already running are not touched.  *sub_index_out = index of the new entry. */
DABGPU_API int dabgpu_msc_add_subchannel(dabgpu_ctx* ctx, int stream, const dabgpu_subchannel* sub, int* sub_index_out);
/* Detach one decoder; the other entries keep their indices and state (no reference analogue: BasicRadio only ever adds). */
DABGPU_API int dabgpu_msc_remove_subchannel(dabgpu_ctx* ctx, int stream, int sub_index);

/* What a sub-channel carries, and so which stage runs on its logical frames after the MSC decode:
 *   STREAM      nothing (the bytes are read with dabgpu_chan_get_msc)
 *   DABPLUS     the DAB+ superframe stage (AAC_Frame_Processor)
 *   PACKET      packet mode without FEC: every logical frame is cut into packets the way basic_data_packet_channel.cpp:49-88
 *               walks it (length from bits 7-6 of byte 0; a tail shorter than 2 bytes or than its packet is dropped)
 *   PACKET_FEC  packet mode with FIG 0/14 FEC scheme 1: the same walk through MSC_Reed_Solomon_Data_Packet_Processor
 *               (msc_reed_solomon_data_packet_processor.cpp:49-258, RS(204,188) per FEC set of 2256 + 9 x 24 bytes)
 * The packet entries report through the sub-channel event log (DABGPU_EV_PACKET / DABGPU_EV_PACKET_FEC records).  Their FEC
 * state (ring of queued packets, last FEC counter) lives across decodes; a fresh entry starts empty.  A set of 2472 bytes spans
 * about 26 decodes at 8 kbit/s, one decode can close several sets at high rates.
 * dabgpu_msc_configure / _add_subchannel are the _ex calls with payload = is_dabplus ? DABPLUS : STREAM.  A packet payload
 * with sc.is_dabplus != 0 gives DABGPU_ERR_INVALID.  An entry whose payload kind changes starts empty. */
enum { DABGPU_PAYLOAD_STREAM = 0, DABGPU_PAYLOAD_DABPLUS = 1, DABGPU_PAYLOAD_PACKET = 2, DABGPU_PAYLOAD_PACKET_FEC = 3 };
typedef struct {
    dabgpu_subchannel sc;
    int payload;         /* DABGPU_PAYLOAD_* */
} dabgpu_subchannel_ex;
DABGPU_API int dabgpu_msc_configure_ex(dabgpu_ctx* ctx, int stream, const dabgpu_subchannel_ex* subs, int n_subs);
DABGPU_API int dabgpu_msc_add_subchannel_ex(dabgpu_ctx* ctx, int stream, const dabgpu_subchannel_ex* sub, int* sub_index_out);

/* BasicRadio::Process: one frame of nb_frame_bits int8 per stream, stream i at frames_host + i*stride.  DABGPU_ERR_OVERFLOW when
 * the frame ring of a stream is full of frames that were not channel-decoded yet (the reference's ThreadedRingBuffer blocks its
 * producer in that case, src/radio_block.cpp:20-44). */
DABGPU_API int dabgpu_softbits_push(dabgpu_ctx* ctx, const int8_t* frames_host, size_t stream_stride_bytes,
                                    int first_stream, int n_streams);

/* ---------------------------------------------------------------------------------------------
 * Self-configuration from the FIC (host only, no GPU work): the FIG 0/1, 0/2, 0/3 and 0/14 subset of
 *   FIG_Processor::ProcessFIB          dab/fic/fig_processor.cpp:94-152, 302-551
 *   Radio_FIG_Handler                  dab/radio_fig_handler.cpp:35-214, 474-481
 *   DAB_Database_Updater (first value of a field wins, required-field masks)  dab/database/dab_database_updater.cpp:94-228
 *   BasicRadio::UpdateAfterProcessing  basic_radio/basic_radio.cpp:83-154 (which sub-channels get a decoder)
 * implemented in sdrplusplus-dab-radio-plugin_b200/host/fic_autoconfig.hpp.
 * ------------------------------------------------------------------------------------------- */
typedef struct dabgpu_autocfg dabgpu_autocfg;
DABGPU_API dabgpu_autocfg* dabgpu_autocfg_create(void);
DABGPU_API void dabgpu_autocfg_destroy(dabgpu_autocfg* a);
/* n_fibs FIBs of `stride` bytes each (30 data bytes are read); crc_ok may be NULL (all valid).  Returns the number of
 * FIBs that changed the database, or a negative dabgpu_status. */
DABGPU_API int dabgpu_autocfg_push_fibs(dabgpu_autocfg* a, const uint8_t* fibs, int n_fibs, size_t stride, const uint8_t* crc_ok);
/* Database dump, rows of int32.  Sub-channels: id, start, length, is_uep, uep_index, eep_level, eep_type (255 = unset),
 * fec_scheme (255 = unset), is_complete.  Components: service id, id type (0 = 16 bit, 1 = 32 bit), component id,
 * sub-channel, global id, transport mode, audio type, data type, packet address, is_complete. */
#define DABGPU_AUTOCFG_SUB_COLS 9
#define DABGPU_AUTOCFG_COMP_COLS 10
DABGPU_API int dabgpu_autocfg_dump(dabgpu_autocfg* a, int32_t* subs, int subs_cap_rows, int* n_subs, int32_t* comps, int comps_cap_rows, int* n_comps);
/* The sub-channels BasicRadio would attach an audio decoder to, in database order; ids[i] = SubChId of out[i]. */
DABGPU_API int dabgpu_autocfg_runnable(dabgpu_autocfg* a, dabgpu_subchannel* out, uint8_t* ids, int cap, int* n_out);
/* BasicRadio::UpdateAfterProcessing: dabgpu_msc_add_subchannel(ctx, stream, ...) for every sub-channel that became runnable since
 * the last call; running decoders are not touched.  Sub-channels the context rejects (invalid range / profile) are skipped for
 * good and do not block the others.  Returns 1 if a decoder was added, 0 if nothing changed, negative on error.  One autocfg
 * object serves one (ctx, stream) pair.  dabgpu_autocfg_applied: SubChId of every sub_index it created, in order. */
DABGPU_API int dabgpu_autocfg_apply(dabgpu_autocfg* a, dabgpu_ctx* ctx, int stream);
DABGPU_API int dabgpu_autocfg_applied(dabgpu_autocfg* a, uint8_t* ids, int cap, int* n_out);

/* ---------------------------------------------------------------------------------------------
 * Capture file formats of the reference's tools (host only): raw IQ in the reader modes of
 *   get_iq_file_reader_from_mode_string   vendor/DAB-Radio/examples/app_helpers/app_iq_readers.h:107-159
 *   QuantisedIQ<T>::to_c32 / QuantisedIQToFloatIQ<T>::read                          app_iq_readers.h:19-87
 * and hard-byte <-> soft-bit frames
 *   convert_viterbi_bits_to_bytes / convert_viterbi_bytes_to_bits   app_helpers/app_viterbi_convert_block.h:12-44
 * implemented in sdrplusplus-dab-radio-plugin_b200/host/capture_formats.hpp.  "raw_u8" and c32 can be fed to
 * dabgpu_ofdm_process directly; the other modes are converted to c32 here, like the reference's readers do.
 * ------------------------------------------------------------------------------------------- */
/* mode: "raw_u8", "raw_s8", "raw_s16l", "raw_s16b", "raw_u16l", "raw_u16b", "raw_s32l", "raw_s32b", "raw_u32l", "raw_u32b",
 * "raw_f32l", "raw_f32b", "raw_f64l", "raw_f64b".  Writes interleaved float I,Q; *n_floats = components converted. */
DABGPU_API int dabgpu_iq_convert(const char* mode, const void* raw, size_t n_bytes, float* out_c32, size_t out_cap_floats, size_t* n_floats);
DABGPU_API int dabgpu_softbits_to_bytes(const int8_t* bits, size_t n_bits, uint8_t* bytes);   /* n_bits multiple of 8 */
DABGPU_API int dabgpu_bytes_to_softbits(const uint8_t* bytes, size_t n_bytes, int8_t* bits);

/* Decodes, for every stream in [first, first+n), the oldest frame in its ring that has not been
 * channel-decoded yet (streams without one are skipped).  Results stay on the device until fetched.
 * A stream whose decoder fell further behind than the ring keeps history for (frame_slots minus the 16-CIF history minus two
 * frames of margin) skips to its newest frame and restarts its time de-interleavers empty; the skipped frames are counted in
 * dabgpu_counters.frames_dropped.  Stale ring slots are never decoded. */
DABGPU_API int dabgpu_chan_decode(dabgpu_ctx* ctx, int first_stream, int n_streams);
/* dabgpu_chan_decode runs on a CUDA stream of its own so that it overlaps the next OFDM stage.  Every getter of this library
 * joins it implicitly; callers that queue their own work or events on dabgpu_cuda_stream() call this (non-blocking) first. */
DABGPU_API int dabgpu_chan_join(dabgpu_ctx* ctx);

/* Result of the last dabgpu_chan_decode for one stream. */
typedef struct {
    int decoded;             /* 1 if a frame of this stream was decoded by the last call */
    int frame_index;         /* index of that frame since context creation */
} dabgpu_chan_status;
DABGPU_API int dabgpu_chan_get_status(dabgpu_ctx* ctx, int stream, dabgpu_chan_status* out);
/* fibs_host: nb_cifs*nb_fibs_per_cif*32 bytes (30 data + 2 CRC, descrambled); crc_ok: one byte per FIB */
DABGPU_API int dabgpu_chan_get_fic(dabgpu_ctx* ctx, int stream, uint8_t* fibs_host, uint8_t* crc_ok);
/* out_host: nb_cifs * bytes_per_cif decoded+descrambled bytes; valid[c] = 0 while the 16-CIF
 * deinterleaver of this sub-channel is still filling (DecodeCIF returns an empty span) */
DABGPU_API int dabgpu_chan_get_msc(dabgpu_ctx* ctx, int stream, int sub_index, uint8_t* out_host, size_t out_cap,
                                   uint8_t* valid, int* bytes_per_cif);

/* Sub-channel event log (DAB+ or packet records) of the last decoded frame.  A DAB+ entry reports the superframe events in the
 * order AAC_Frame_Processor would have fired its observers (OnFirecodeError/OnRSError/OnSuperFrameHeader/OnAccessUnitCRCError/
 * OnAccessUnit).  A packet entry (DABGPU_PAYLOAD_PACKET / _PACKET_FEC) reports, in order:
 *   DABGPU_EV_PACKET      one per packet the processor hands on (the adapter's callback): a = is_corrected, b = crc_ok (CRC16-CCITT
 *                         of packet[:-2], init 0xFFFF, inverted, equals the last two bytes big-endian; EN 300 401 5.3.2),
 *                         c = 10-bit packet address, d = 0; payload = the whole packet (24, 48, 72 or 96 bytes).  Without FEC
 *                         every packet has is_corrected = 0.
 *   DABGPU_EV_PACKET_FEC  each time an FEC set ends, just before the packets it releases (also when it releases none):
 *                         a = 1 when the 12 rows were decoded, then b = rows decoded, c = rows uncorrectable, d = sum of the
 *                         decoded rows' error counts; a = 0 when the set was abandoned (broken FEC counter or incomplete ring),
 *                         then b = c = d = 0.  No payload. */
enum { DABGPU_EV_FIRECODE_ERROR = 1, DABGPU_EV_RS_ERROR = 2, DABGPU_EV_SUPERFRAME_HEADER = 3,
       DABGPU_EV_AU_CRC_ERROR = 4, DABGPU_EV_ACCESS_UNIT = 5, DABGPU_EV_PACKET = 6, DABGPU_EV_PACKET_FEC = 7 };
typedef struct { int32_t type, a, b, c, d, n_bytes; } dabgpu_event_header;  /* followed by n_bytes payload padded to 4 */
DABGPU_API int dabgpu_chan_get_dabplus_events(dabgpu_ctx* ctx, int stream, int sub_index, uint8_t* log_host,
                                              size_t log_cap, size_t* log_bytes);

/* Sub-channel event logs (DAB+ or packet records) of every sub-channel of streams [first, first+n) at once, packed on the GPU.
 * index_host: [n][max_subchannels][2] int32 = {byte offset into log_host, byte length}.  The log of (stream, sub) is
 * byte-identical to what dabgpu_chan_get_dabplus_events(stream, sub) returns after the same decode: dabgpu_event_header
 * records + payload padded to 4.  Length 0 = no events, a STREAM sub-channel, or an unused index.  Where the logs sit inside
 * log_host is not part of the contract: read it through the index.
 *
 * A packet entry with A = nb_cifs x bytes-per-CIF arriving per decode hands on at most 2472 + A bytes of packets (its FEC ring
 * plus what arrived) and ends at most A / 24 FEC sets, so its log stays below 24 x (2472 + A) / 24 + (2472 + A) + 24 x (A / 24 + 1)
 * bytes; dabgpu_dabplus_out_bound counts that for it.
 *
 * dabgpu_dabplus_out_bound: the log_cap one decode of those streams can never exceed.  It follows from the sub-channel tables
 * (active DAB+ and packet entries and their bytes per CIF): a decode runs one frame of at most 4 CIFs per stream and a superframe takes 5,
 * so each (stream, sub) fires at most 7 events and 5 x bytes-per-CIF of AU payload.  It changes with dabgpu_msc_configure /
 * _add_subchannel / _remove_subchannel.  A log_cap below it gives DABGPU_ERR_OVERFLOW; NULL log_host or index_host gives
 * DABGPU_ERR_INVALID.  Both are refused before anything is queued and leave the context as it was.
 *
 * dabgpu_chan_get_dabplus_all: the output of the last dabgpu_chan_decode that covered each stream; synchronises the context.
 * dabgpu_submit_ex / dabgpu_wideband_submit_ex: dabgpu_submit / dabgpu_wideband_submit that also copy the DAB+ output of the
 * ticket's channel decode into *dabplus (which needs run_chan_decode != 0, else DABGPU_ERR_INVALID).  The buffers must stay
 * valid until the ticket was waited for and be pinned for the copy to overlap.  dabplus = NULL is exactly dabgpu_submit /
 * dabgpu_wideband_submit.  The struct is read during the call only. */
typedef struct {
    uint8_t* log_host;
    size_t log_cap;
    int32_t* index_host;
} dabgpu_dabplus_out;
DABGPU_API int dabgpu_dabplus_out_bound(dabgpu_ctx* ctx, int first_stream, int n_streams, size_t* log_bytes);
DABGPU_API int dabgpu_chan_get_dabplus_all(dabgpu_ctx* ctx, int first_stream, int n_streams, const dabgpu_dabplus_out* out);
DABGPU_API int dabgpu_submit_ex(dabgpu_ctx* ctx, const dabgpu_step* step, const dabgpu_dabplus_out* dabplus, uint64_t* ticket);
DABGPU_API int dabgpu_wideband_submit_ex(dabgpu_wideband* w, const dabgpu_step* step, const dabgpu_dabplus_out* dabplus,
                                         uint64_t* ticket);

/* Stand-alone AAC_Frame_Processor (dab/audio/aac_frame_processor.h:37-82): one object per DAB+ sub-channel that is
 * fed decoded logical frames from the host.  process() consumes one logical frame (MSC_Decoder::DecodeCIF output) and
 * returns the observer events it fired, in order, in the same flat log format as dabgpu_chan_get_dabplus_events. */
typedef struct dabgpu_dabplus dabgpu_dabplus;
DABGPU_API int dabgpu_dabplus_open(dabgpu_ctx* ctx, dabgpu_dabplus** out);
DABGPU_API void dabgpu_dabplus_close(dabgpu_ctx* ctx, dabgpu_dabplus* p);
DABGPU_API int dabgpu_dabplus_process(dabgpu_ctx* ctx, dabgpu_dabplus* p, const uint8_t* frame_host, int n_bytes, uint8_t* log_host,
                                      size_t log_cap, size_t* log_bytes);

/* Reed_Solomon_Decoder::Decode batched (reed_solomon_decoder.h:18-26; GF(2^8)/0x11D, fcr 0, prim 1):
 * n_codewords codewords of (255-pad) bytes each, corrected in place; counts[i] = return value of
 * Decode (-1 = uncorrectable), positions (optional) = nroots ints per codeword (error locations incl. pad). */
DABGPU_API int dabgpu_rs_decode(dabgpu_ctx* ctx, uint8_t* codewords_host, int n_codewords, int nroots, int pad,
                                int* counts_host, int* positions_host);

/* Packet-mode FEC (ETSI EN 300 401 5.3.5), the Reed-Solomon step of
 * MSC_Reed_Solomon_Data_Packet_Processor::PerformReedSolomonCorrection (dab/msc/msc_reed_solomon_data_packet_processor.cpp:200-240):
 * n_frames FEC frames of DABGPU_PACKET_FEC_FRAME_BYTES each = the 2256-byte application data table (the data packets in
 * transport order) followed by the 192-byte RS data table (data fields of the nine FEC packets, headers and the six
 * padding bytes removed).  The 12 rows of every frame are decoded as RS(204,188) (16 roots, shortened by 51) and the
 * application data table is corrected in place; the RS data table is left as received, like the reference.
 * row_counts (optional) = 12 ints per frame, the return value of Reed_Solomon_Decoder::Decode per row (-1 = uncorrectable). */
#define DABGPU_PACKET_FEC_FRAME_BYTES 2448
#define DABGPU_PACKET_FEC_ROWS 12
DABGPU_API int dabgpu_packet_fec_decode(dabgpu_ctx* ctx, uint8_t* frames_host, int n_frames, int* row_counts_host);

/* Whole-chain convenience for throughput runs: OFDM advance + channel decode of the frames produced. */
typedef struct {
    uint64_t frames_demodulated;   /* totals since context creation */
    uint64_t frames_channel_decoded;
    uint64_t fibs_crc_ok, fibs_total;
    uint64_t msc_bytes_decoded;
    uint64_t superframes_ok, superframes_rs_fail, superframes_firecode_fail;
    uint64_t au_ok, au_crc_fail;
    uint64_t frames_dropped;       /* frames the channel decoder skipped because it fell behind the frame ring (see dabgpu_chan_decode) */
} dabgpu_counters;
DABGPU_API int dabgpu_get_counters(dabgpu_ctx* ctx, dabgpu_counters* out);

#ifdef __cplusplus
}
#endif
#endif /* DABGPU_H */
