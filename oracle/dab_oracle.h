/* oracle/dab_oracle.h -- TEST INFRASTRUCTURE, not product code.
 *
 * Plain-C CPU restatement of the DAB receive hot path of the reference
 * (williamyang98/SDRPlusPlus-DAB-Radio-Plugin, vendor/DAB-Radio).  It exists so that the CUDA
 * path can be checked on a box where /root/reference is absent, and it is itself pinned against
 * the reference's own code (oracle/_ref/libdabref.so, built by oracle/Makefile from the
 * unmodified sources) by tests/test_oracle_vs_ref.py.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may use this library.
 * Each function cites the reference file:line it follows; paths are relative to
 * /root/reference/vendor/DAB-Radio/ (VIT = vendor/viterbi_decoder/include/viterbi).
 *
 * Parity status:
 *   integer stages (depuncture, Viterbi, traceback, descramble, CRC, deinterleave, RS, superframe)
 *     -> pinned bit-exact against the reference build "x86 AVX2 u16" (tie => decision 1, saturating u16).
 *   OFDM (float32) -> pinned within max|delta| <= 1 soft-bit LSB; FFT boundary itself is unpinned in the
 *     reference (FFTW3 is an external, absent dependency; both oracles use their own FFT).
 */
#ifndef DAB_ORACLE_H
#define DAB_ORACLE_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* ---- tables ---- */
void dabo_pi_counts(int pi, uint8_t out8[8]);                       /* puncture_codes.h:42-67 */
int  dabo_eep_segments(int length, int level, int type_b, int seg_pi[3], int seg_bits[3]);
int  dabo_uep_segments(int index, int seg_pi[5], int seg_bits[5]);  /* returns number of segments */
int  dabo_ofdm_params(int mode, int out6[6]);  /* frame_symbols, symbol_period, null_period, cyclic_prefix, fft, carriers */
int  dabo_carrier_map(int nb_fft, int nb_carriers, int* out);
int  dabo_prs_fft(int mode, float* out_interleaved, int nb_fft);

/* ---- integer chain ---- */
int  dabo_vit_decode(const int8_t* soft, int n_soft, const int* seg_pi, const int* seg_bits, int n_seg,
                     uint8_t* out_bytes, int n_out_bytes, uint64_t* path_error);
void dabo_scrambler_bytes(uint8_t* out, int n);
uint16_t dabo_crc16(const uint8_t* data, int n, uint16_t poly, uint16_t init, uint16_t xorout);
int  dabo_fic_decode_group(const int8_t* bits2304, uint8_t out96[96], int crc_ok[3]);

typedef struct dabo_msc dabo_msc;
dabo_msc* dabo_msc_create(int start_address, int length, int is_uep, int uep_index, int eep_level, int eep_type_b);
void dabo_msc_destroy(dabo_msc*);
int  dabo_msc_decode_cif(dabo_msc*, const int8_t* cif_bits, int n_bits, uint8_t* out, int out_cap);

int  dabo_rs_decode(int nroots, int pad, uint8_t* data, int* eras_pos);

typedef struct dabo_aac dabo_aac;
dabo_aac* dabo_aac_create(void);
void dabo_aac_destroy(dabo_aac*);
/* same flat event log format as oracle/ref_harness.cpp (EV_* codes) */
int  dabo_aac_process(dabo_aac*, const uint8_t* frame, int n, uint8_t* log_out, int log_cap);

/* ---- OFDM ---- */
typedef struct dabo_ofdm dabo_ofdm;
/* OFDM_Demod_Config (ofdm_demodulator.h:24-45), fields in the order of dabgpu_ofdm_config */
typedef struct {
    float signal_l1_update_beta;
    int   signal_l1_nb_samples;
    int   signal_l1_nb_decimate;
    float null_thresh_start;
    float null_thresh_end;
    float fine_freq_update_beta;
    int   is_coarse_freq_correction;
    float max_coarse_freq_correction_norm;
    float coarse_freq_slow_beta;
    float impulse_peak_threshold_db;
    float impulse_peak_distance_probability;
} dabo_ofdm_config;
dabo_ofdm* dabo_ofdm_create(int mode);
/* OFDM_Demod::GetConfig() = *cfg: in force from the next process call on */
void dabo_ofdm_set_config(dabo_ofdm*, const dabo_ofdm_config* cfg);
void dabo_ofdm_destroy(dabo_ofdm*);
int  dabo_ofdm_frame_bits(const dabo_ofdm*);
void dabo_ofdm_process_c32(dabo_ofdm*, const float* iq, int n_samples);
void dabo_ofdm_process_u8(dabo_ofdm*, const uint8_t* iq, int n_samples);
int  dabo_ofdm_pop_frame(dabo_ofdm*, int8_t* out, float* coarse_fine2, int* time_offset);
void dabo_ofdm_get_state(const dabo_ofdm*, int* state4, float* fstate3);
void dabo_ofdm_keep_frames(dabo_ofdm*, int keep);
void dabo_fft(float* data_interleaved, int n, int inverse);   /* in place, unnormalised */

/* ---- timing helpers for bench.py cpu_baseline (kind "port") ---- */
double dabo_time_ofdm_u8(int mode, const uint8_t* iq, long n_samples, int block_size, int repeat, int* frames_out);

#ifdef __cplusplus
}
#endif
#endif
