// oracle/ref_harness.cpp -- TEST INFRASTRUCTURE, not product code.
//
// C-ABI driver around the UNMODIFIED reference classes, compiled in place from
// /root/reference by oracle/Makefile into oracle/_ref/libdabref.so.  It is the
// checker that pins oracle/dab_oracle.c (the CPU restatement) and the CUDA path.
// Nothing here is linked into the product library.
//
// Reference classes driven (paths relative to /root/reference/vendor/DAB-Radio/src):
//   DAB_Viterbi_Decoder   dab/algorithms/dab_viterbi_decoder.h:12-45
//   AdditiveScrambler     dab/algorithms/additive_scrambler.h:10-36
//   FIC_Decoder           dab/fic/fic_decoder.h
//   MSC_Decoder           dab/msc/msc_decoder.h:19-38
//   CIF_Deinterleaver     dab/msc/cif_deinterleaver.h
//   Reed_Solomon_Decoder  dab/algorithms/reed_solomon_decoder.h
//   AAC_Frame_Processor   dab/audio/aac_frame_processor.h:37-82
//   OFDM_Demod            ofdm/ofdm_demodulator.h:47-160
//
// OFDM determinism (SURVEY.md H2/H3): the reference's reader thread keeps
// consuming samples (and runs the next frame's coarse/fine sync) while the
// pipeline thread is still demodulating the frame just completed, so the fine
// frequency offset seen by either side is timing dependent.  The "serial" driver
// below re-states the 30-line dispatcher of OFDM_Demod::Process
// (ofdm_demodulator.cpp:235-275) using the class's own private methods and
// waits for the On_OFDM_Frame callback right after ReadSymbols completes a
// frame.  Every arithmetic routine that runs is the reference's own code.

#include <stddef.h>
#include <stdint.h>
#include <string.h>
#include <atomic>
#include <chrono>
#include <complex>
#include <condition_variable>
#include <cstdio>
#include <functional>
#include <memory>
#include <mutex>
#include <thread>
#include <unordered_map>
#include <vector>
#include <optional>
#include <string>
#include <fmt/format.h>

// private access for the deterministic OFDM driver only (layout is unaffected with GCC)
#define private public
#include "ofdm/ofdm_demodulator.h"
#include "ofdm/ofdm_demodulator_threads.h"
#undef private

#include "ofdm/dab_mapper_ref.h"
#include "ofdm/dab_ofdm_params_ref.h"
#include "ofdm/dab_prs_ref.h"
#include "dab/algorithms/additive_scrambler.h"
#include "dab/algorithms/dab_viterbi_decoder.h"
#include "dab/algorithms/reed_solomon_decoder.h"
#include "dab/audio/aac_frame_processor.h"
#include "dab/constants/dab_parameters.h"
#include "dab/constants/puncture_codes.h"
#include "dab/constants/subchannel_protection_tables.h"
#include "dab/database/dab_database_entities.h"
#include "dab/fic/fic_decoder.h"
#include "dab/msc/cif_deinterleaver.h"
#include "dab/msc/msc_decoder.h"
#include "dab/msc/msc_reed_solomon_data_packet_processor.h"
#include "viterbi_config.h"

#define API extern "C" __attribute__((visibility("default")))

// ---------------------------------------------------------------------------------------------
// Build information
// ---------------------------------------------------------------------------------------------
API const char* ref_build_info() {
#if defined(__AVX2__)
    return "reference sources; DAB_VITERBI_DECODER=x86 AVX2 u16; apply_pll=AVX"
#if defined(__FMA__)
           "+FMA"
#endif
           "; FFT=oracle/fft_shim.cpp (FFTW3 absent)";
#else
    return "reference sources; non-AVX2 build (NOT the pinned semantics)";
#endif
}

// ---------------------------------------------------------------------------------------------
// Viterbi: depuncture segments + chainback through DAB_Viterbi_Decoder
// ---------------------------------------------------------------------------------------------
struct RefVit { DAB_Viterbi_Decoder dec; };

API void* ref_vit_create() { return new RefVit(); }
API void ref_vit_destroy(void* h) { delete (RefVit*)h; }

// seg_pi[i] in 1..24 selects PI_TABLE row, 0 selects the tail code PI_X.
// seg_bits[i] = requested mother-code symbols (multiple of 4).
// Returns number of punctured symbols consumed, or -1 on bad arguments.
API int ref_vit_decode(void* h, const int8_t* soft, int n_soft,
                       const int* seg_pi, const int* seg_bits, int n_seg,
                       uint8_t* out_bytes, int n_out_bytes, uint64_t* path_error) {
    auto& dec = ((RefVit*)h)->dec;
    int total_steps = 0;
    for (int i = 0; i < n_seg; i++) total_steps += seg_bits[i]/4;
    if (n_out_bytes*8 + 6 > total_steps) return -1;
    dec.set_traceback_length(size_t(total_steps));
    dec.reset();
    tcb::span<const viterbi_bit_t> buf(soft, size_t(n_soft));
    int consumed = 0;
    for (int i = 0; i < n_seg; i++) {
        tcb::span<const uint8_t> code = (seg_pi[i] == 0) ? tcb::span<const uint8_t>(PI_X) : GetPunctureCode(seg_pi[i]);
        const size_t N = dec.update(buf, code, size_t(seg_bits[i]));
        buf = buf.subspan(N);
        consumed += int(N);
    }
    const uint64_t err = dec.chainback({out_bytes, size_t(n_out_bytes)});
    if (path_error) *path_error = err;
    return consumed;
}

// Energy dispersal PRBS bytes (additive_scrambler.h), syncword 0xFFFF
API void ref_scrambler_bytes(uint8_t* out, int n) {
    AdditiveScrambler s;
    s.SetSyncword(0xFFFF);
    s.Reset();
    for (int i = 0; i < n; i++) out[i] = s.Process();
}

// ---------------------------------------------------------------------------------------------
// FIC
// ---------------------------------------------------------------------------------------------
struct RefFic {
    std::unique_ptr<FIC_Decoder> dec;
    std::vector<uint8_t> fibs;   // 30 bytes each, in emission order
    int nb_fibs = 0;
};

API void* ref_fic_create(int nb_encoded_bits, int nb_fibs_per_group) {
    auto* r = new RefFic();
    r->dec = std::make_unique<FIC_Decoder>(size_t(nb_encoded_bits), size_t(nb_fibs_per_group));
    r->dec->OnFIB().Attach([r](tcb::span<const uint8_t> buf) {
        r->fibs.insert(r->fibs.end(), buf.begin(), buf.end());
        r->nb_fibs++;
    });
    return r;
}
API void ref_fic_destroy(void* h) { delete (RefFic*)h; }

// Decodes one FIB group; copies the CRC-valid FIBs (30 bytes each) in emission order.
API int ref_fic_decode_group(void* h, const int8_t* bits, int n_bits, int cif_index, uint8_t* fibs_out, int fibs_cap) {
    auto* r = (RefFic*)h;
    r->fibs.clear();
    r->nb_fibs = 0;
    r->dec->DecodeFIBGroup({bits, size_t(n_bits)}, size_t(cif_index));
    const int n = (r->nb_fibs < fibs_cap) ? r->nb_fibs : fibs_cap;
    if (n > 0) memcpy(fibs_out, r->fibs.data(), size_t(n)*30);
    return r->nb_fibs;
}

// ---------------------------------------------------------------------------------------------
// MSC sub-channel decoder
// ---------------------------------------------------------------------------------------------
struct RefMsc { std::unique_ptr<MSC_Decoder> dec; };

// UEP_PROTECTION_TABLE row (dab/constants/subchannel_protection_tables.h:21-86): {size CU, bitrate, level, L1..L4, PI1..PI4, padding bits}
API int ref_uep_descriptor(int index, int* out12) {
    if (index < 0 || index >= UEP_PROTECTION_TABLE_SIZE) return -1;
    const UEP_Descriptor& d = UEP_PROTECTION_TABLE[index];
    out12[0] = d.subchannel_size; out12[1] = d.bitrate; out12[2] = d.protection_level;
    for (int i = 0; i < 4; i++) { out12[3 + i] = d.Lx[i]; out12[7 + i] = d.PIx[i]; }
    out12[11] = d.total_padding_bits;
    return 0;
}

API void* ref_msc_create(int start_address, int length, int is_uep, int uep_index, int eep_level, int eep_type_b) {
    Subchannel sc(0);
    sc.start_address = subchannel_addr_t(start_address);
    sc.length = subchannel_size_t(length);
    sc.is_uep = is_uep != 0;
    sc.uep_prot_index = uep_protection_index_t(uep_index);
    sc.eep_prot_level = eep_protection_level_t(eep_level);
    sc.eep_type = eep_type_b ? EEP_Type::TYPE_B : EEP_Type::TYPE_A;
    auto* r = new RefMsc();
    r->dec = std::make_unique<MSC_Decoder>(sc);
    return r;
}
API void ref_msc_destroy(void* h) { delete (RefMsc*)h; }

// Returns decoded byte count (0 while the 16-CIF deinterleaver is filling).
API int ref_msc_decode_cif(void* h, const int8_t* cif_bits, int n_bits, uint8_t* out, int out_cap) {
    auto* r = (RefMsc*)h;
    auto res = r->dec->DecodeCIF({cif_bits, size_t(n_bits)});
    const int n = int(res.size());
    if (n > out_cap) return -n;
    if (n > 0) memcpy(out, res.data(), size_t(n));
    return n;
}

// CIF_Deinterleaver on its own
struct RefDeint { std::unique_ptr<CIF_Deinterleaver> d; int nb_bits; };
API void* ref_deint_create(int nb_bytes) {
    auto* r = new RefDeint();
    r->d = std::make_unique<CIF_Deinterleaver>(nb_bytes);
    r->nb_bits = nb_bytes*8;
    return r;
}
API void ref_deint_destroy(void* h) { delete (RefDeint*)h; }
API int ref_deint_push(void* h, const int8_t* in_bits, int8_t* out_bits) {
    auto* r = (RefDeint*)h;
    r->d->Consume({in_bits, size_t(r->nb_bits)});
    return r->d->Deinterleave({out_bits, size_t(r->nb_bits)}) ? 1 : 0;
}

// ---------------------------------------------------------------------------------------------
// Reed-Solomon (Phil Karn decode_rs_char wrapped by Reed_Solomon_Decoder)
// ---------------------------------------------------------------------------------------------
struct RefRs { std::unique_ptr<Reed_Solomon_Decoder> d; };
API void* ref_rs_create(int symsize, int gfpoly, int fcr, int prim, int nroots, int pad) {
    auto* r = new RefRs();
    r->d = std::make_unique<Reed_Solomon_Decoder>(symsize, gfpoly, fcr, prim, nroots, pad);
    return r;
}
API void ref_rs_destroy(void* h) { delete (RefRs*)h; }
API int ref_rs_decode(void* h, uint8_t* data, int* eras_pos, int no_eras) {
    return ((RefRs*)h)->d->Decode(data, eras_pos, no_eras);
}

// ---------------------------------------------------------------------------------------------
// Packet-mode FEC (MSC_Reed_Solomon_Data_Packet_Processor): callbacks serialised into a flat log
// record: int32 nbytes, int32 is_corrected, then the packet (padded to 4)
// ---------------------------------------------------------------------------------------------
struct RefPktFec {
    MSC_Reed_Solomon_Data_Packet_Processor proc;
    std::vector<uint8_t> log;
};
API void* ref_pktfec_create() {
    auto* r = new RefPktFec();
    r->proc.SetCallback([r](tcb::span<const uint8_t> pkt, bool corrected) {
        const int32_t hdr[2] = {int32_t(pkt.size()), corrected ? 1 : 0};
        const size_t off = r->log.size(), pad = (pkt.size() + 3u) & ~size_t(3);
        r->log.resize(off + sizeof(hdr) + pad, 0);
        memcpy(&r->log[off], hdr, sizeof(hdr));
        if (!pkt.empty()) memcpy(&r->log[off + sizeof(hdr)], pkt.data(), pkt.size());
    });
    return r;
}
API void ref_pktfec_destroy(void* h) { delete (RefPktFec*)h; }
// returns the number of bytes ReadPacket consumed; the callbacks fired by this call are appended to log_out
API long ref_pktfec_read_packet(void* h, const uint8_t* buf, int n, uint8_t* log_out, int log_cap, int* log_bytes) {
    auto* r = (RefPktFec*)h;
    r->log.clear();
    const size_t used = r->proc.ReadPacket({buf, size_t(n)});
    *log_bytes = int(r->log.size());
    if (int(r->log.size()) > log_cap) return -1;
    if (!r->log.empty()) memcpy(log_out, r->log.data(), r->log.size());
    return long(used);
}

// ---------------------------------------------------------------------------------------------
// DAB+ superframe processor: events serialised into a flat int32/byte log
// ---------------------------------------------------------------------------------------------
// event record: int32 type, int32 a, int32 b, int32 c, int32 d, int32 nbytes, then nbytes payload (padded to 4)
enum { EV_FIRECODE_ERROR = 1, EV_RS_ERROR = 2, EV_HEADER = 3, EV_AU_CRC_ERROR = 4, EV_AU = 5 };
struct RefAac {
    AAC_Frame_Processor proc;
    std::vector<uint8_t> log;
    void push(int type, int a, int b, int c, int d, const uint8_t* payload, int nbytes) {
        int32_t hdr[6] = {type, a, b, c, d, nbytes};
        const size_t off = log.size();
        const size_t pad = (size_t(nbytes) + 3u) & ~size_t(3);
        log.resize(off + sizeof(hdr) + pad, 0);
        memcpy(&log[off], hdr, sizeof(hdr));
        if (nbytes > 0) memcpy(&log[off+sizeof(hdr)], payload, size_t(nbytes));
    }
};
API void* ref_aac_create() {
    auto* r = new RefAac();
    r->proc.OnFirecodeError().Attach([r](const int frame, const uint16_t got, const uint16_t calc) {
        r->push(EV_FIRECODE_ERROR, frame, got, calc, 0, nullptr, 0);
    });
    r->proc.OnRSError().Attach([r](const int idx, const int total) {
        r->push(EV_RS_ERROR, idx, total, 0, 0, nullptr, 0);
    });
    r->proc.OnSuperFrameHeader().Attach([r](SuperFrameHeader hdr) {
        r->push(EV_HEADER, int(hdr.sampling_rate), (hdr.is_parametric_stereo ? 1 : 0) | (hdr.is_spectral_band_replication ? 2 : 0) | (hdr.is_stereo ? 4 : 0),
                int(hdr.mpeg_surround), 0, nullptr, 0);
    });
    r->proc.OnAccessUnitCRCError().Attach([r](const int au, const int total, const uint16_t got, const uint16_t calc) {
        r->push(EV_AU_CRC_ERROR, au, total, got, calc, nullptr, 0);
    });
    r->proc.OnAccessUnit().Attach([r](const int au, const int total, tcb::span<uint8_t> buf) {
        r->push(EV_AU, au, total, 0, 0, buf.data(), int(buf.size()));
    });
    return r;
}
API void ref_aac_destroy(void* h) { delete (RefAac*)h; }
// Feed one logical frame; returns number of log bytes produced by this call (copied to log_out if it fits)
API int ref_aac_process(void* h, const uint8_t* frame, int n, uint8_t* log_out, int log_cap) {
    auto* r = (RefAac*)h;
    r->log.clear();
    r->proc.Process({frame, size_t(n)});
    const int L = int(r->log.size());
    if (L > 0 && L <= log_cap) memcpy(log_out, r->log.data(), size_t(L));
    return L;
}
// Access to the (RS corrected) superframe buffer is private in the reference; expose state needed by tests
API int ref_aac_superframe_size(void* h) {
    (void)h; return 0;
}

// ---------------------------------------------------------------------------------------------
// Tables
// ---------------------------------------------------------------------------------------------
API int ref_ofdm_params(int mode, int* out6) {
    try {
        const auto p = get_DAB_OFDM_params(mode);
        out6[0] = int(p.nb_frame_symbols); out6[1] = int(p.nb_symbol_period); out6[2] = int(p.nb_null_period);
        out6[3] = int(p.nb_cyclic_prefix); out6[4] = int(p.nb_fft); out6[5] = int(p.nb_data_carriers);
        return 0;
    } catch (...) { return -1; }
}
API int ref_prs_fft(int mode, float* out_interleaved, int nb_fft) {
    try {
        std::vector<std::complex<float>> buf(static_cast<size_t>(nb_fft));
        get_DAB_PRS_reference(mode, buf);
        memcpy(out_interleaved, buf.data(), sizeof(float)*2*size_t(nb_fft));
        return 0;
    } catch (...) { return -1; }
}
API int ref_carrier_map(int nb_fft, int nb_carriers, int* out) {
    std::vector<int> m(static_cast<size_t>(nb_carriers));
    get_DAB_mapper_ref(m, size_t(nb_fft));
    memcpy(out, m.data(), sizeof(int)*size_t(nb_carriers));
    return 0;
}
API int ref_dab_params(int mode, int* out13) {
    try {
        const auto p = get_dab_parameters(mode);
        const int v[13] = {p.nb_frame_bits, p.nb_symbols, p.nb_fic_symbols, p.nb_msc_symbols, p.nb_fibs, p.nb_cifs, p.nb_fibs_per_cif,
                           p.nb_sym_bits, p.nb_fic_bits, p.nb_msc_bits, p.nb_fib_bits, p.nb_fib_cif_bits, p.nb_cif_bits};
        memcpy(out13, v, sizeof(v));
        return 0;
    } catch (...) { return -1; }
}

// ---------------------------------------------------------------------------------------------
// OFDM demodulator
// ---------------------------------------------------------------------------------------------
struct RefOfdm {
    OFDM_Params params;
    std::vector<std::complex<float>> prs;
    std::vector<int> mapper;
    std::unique_ptr<OFDM_Demod> demod;
    size_t frame_bits = 0;
    // frames delivered by the callback (coordinator thread)
    std::mutex mtx;
    std::condition_variable cv;
    std::vector<std::vector<int8_t>> frames;
    // snapshot of sync state taken inside the callback: coarse, fine, fine_time_offset
    std::vector<float> frame_coarse, frame_fine;
    std::vector<int> frame_time_offset;
    size_t frames_done = 0;       // callbacks received
    size_t frames_triggered = 0;  // serial driver: frames handed to the coordinator
    size_t frames_popped = 0;
    bool keep_frames = true;
    std::vector<std::complex<float>> scratch;
};

API void* ref_ofdm_create(int mode, int nb_threads) {
    auto* r = new RefOfdm();
    try {
        r->params = get_DAB_OFDM_params(mode);
        r->prs.resize(r->params.nb_fft);
        get_DAB_PRS_reference(mode, r->prs);
        r->mapper.resize(r->params.nb_data_carriers);
        get_DAB_mapper_ref(r->mapper, r->params.nb_fft);
    } catch (...) { delete r; return nullptr; }
    r->demod = std::make_unique<OFDM_Demod>(r->params, r->prs, r->mapper, nb_threads);
    r->frame_bits = (r->params.nb_frame_symbols-1)*r->params.nb_data_carriers*2;
    r->demod->On_OFDM_Frame().Attach([r](tcb::span<const viterbi_bit_t> bits) {
        std::unique_lock<std::mutex> lock(r->mtx);
        if (r->keep_frames) {
            r->frames.emplace_back(bits.begin(), bits.end());
            r->frame_coarse.push_back(r->demod->GetCoarseFrequencyOffset());
            r->frame_fine.push_back(r->demod->GetFineFrequencyOffset());
            r->frame_time_offset.push_back(r->demod->GetFineTimeOffset());
        }
        r->frames_done++;
        r->cv.notify_all();
    });
    return r;
}
API void ref_ofdm_destroy(void* h) { delete (RefOfdm*)h; }
API void ref_ofdm_keep_frames(void* h, int keep) { ((RefOfdm*)h)->keep_frames = keep != 0; }
API int ref_ofdm_frame_bits(void* h) { return int(((RefOfdm*)h)->frame_bits); }

// Deterministic driver: same dispatch as OFDM_Demod::Process (ofdm_demodulator.cpp:241-274)
// plus a wait for the frame callback immediately after a frame is handed to the coordinator.
static void process_serial(RefOfdm* r, tcb::span<const std::complex<float>> buf) {
    auto& d = *r->demod;
    d.UpdateSignalAverage(buf);
    const size_t N = buf.size();
    size_t curr = 0;
    while (curr < N) {
        auto* block = &buf[curr];
        const size_t remain = N - curr;
        const auto state_before = d.m_state;
        switch (d.m_state) {
        case OFDM_Demod::State::FINDING_NULL_POWER_DIP:  curr += d.FindNullPowerDip({block, remain}); break;
        case OFDM_Demod::State::READING_NULL_AND_PRS:    curr += d.ReadNullPRS({block, remain}); break;
        case OFDM_Demod::State::RUNNING_COARSE_FREQ_SYNC:curr += d.RunCoarseFreqSync({block, remain}); break;
        case OFDM_Demod::State::RUNNING_FINE_TIME_SYNC:  curr += d.RunFineTimeSync({block, remain}); break;
        case OFDM_Demod::State::READING_SYMBOLS:         curr += d.ReadSymbols({block, remain}); break;
        }
        if (state_before == OFDM_Demod::State::READING_SYMBOLS && d.m_state == OFDM_Demod::State::READING_NULL_AND_PRS) {
            r->frames_triggered++;
            std::unique_lock<std::mutex> lock(r->mtx);
            r->cv.wait(lock, [r]() { return r->frames_done >= r->frames_triggered; });
        }
    }
}

// iq: interleaved float re,im ; serial != 0 selects the deterministic driver
API void ref_ofdm_process_c32(void* h, const float* iq, int n_samples, int serial) {
    auto* r = (RefOfdm*)h;
    tcb::span<const std::complex<float>> buf(reinterpret_cast<const std::complex<float>*>(iq), size_t(n_samples));
    if (serial) process_serial(r, buf); else r->demod->Process(buf);
}

// u8 IQ converted exactly like QuantisedIQToFloatIQ<uint8_t>::read
// (examples/app_helpers/app_iq_readers.h:23-43, 72-87): (u8 - 127.5f) * (1.0f/127.5f)
API void ref_ofdm_process_u8(void* h, const uint8_t* iq, int n_samples, int serial) {
    auto* r = (RefOfdm*)h;
    r->scratch.resize(size_t(n_samples));
    constexpr float BIAS = 127.5f;
    constexpr float scale = 1.0f/127.5f;
    for (int i = 0; i < n_samples; i++) {
        const float re = float(iq[2*i+0]) - BIAS;
        const float im = float(iq[2*i+1]) - BIAS;
        r->scratch[size_t(i)] = std::complex<float>(re*scale, im*scale);
    }
    tcb::span<const std::complex<float>> buf(r->scratch);
    if (serial) process_serial(r, buf); else r->demod->Process(buf);
}

// Free-running mode: wait until every frame handed over so far has been delivered
API void ref_ofdm_flush(void* h) {
    auto* r = (RefOfdm*)h;
    // the coordinator sets is_end before it notifies observers, so poll the callback count against frames_read
    r->demod->m_coordinator->WaitEnd();
    r->demod->m_coordinator->SignalEnd();
    for (int i = 0; i < 2000; i++) {
        {
            std::unique_lock<std::mutex> lock(r->mtx);
            if (int(r->frames_done) >= r->demod->GetTotalFramesRead()) return;
        }
        std::this_thread::sleep_for(std::chrono::milliseconds(1));
    }
}

API int ref_ofdm_frames_available(void* h) {
    auto* r = (RefOfdm*)h;
    std::unique_lock<std::mutex> lock(r->mtx);
    return int(r->frames.size() - r->frames_popped);
}
// pops the oldest frame; info3 = {coarse, fine} as floats bit-cast is avoided: separate arrays
API int ref_ofdm_pop_frame(void* h, int8_t* out, float* coarse_fine2, int* time_offset) {
    auto* r = (RefOfdm*)h;
    std::unique_lock<std::mutex> lock(r->mtx);
    if (r->frames_popped >= r->frames.size()) return 0;
    const size_t i = r->frames_popped++;
    memcpy(out, r->frames[i].data(), r->frames[i].size());
    if (coarse_fine2) { coarse_fine2[0] = r->frame_coarse[i]; coarse_fine2[1] = r->frame_fine[i]; }
    if (time_offset) *time_offset = r->frame_time_offset[i];
    std::vector<int8_t>().swap(r->frames[i]);
    return 1;
}
// state: {state, frames_read, frames_desync, fine_time_offset}; fstate: {signal_avg, coarse, fine}
API void ref_ofdm_get_state(void* h, int* state4, float* fstate3) {
    auto& d = *((RefOfdm*)h)->demod;
    state4[0] = int(d.GetState());
    state4[1] = d.GetTotalFramesRead();
    state4[2] = d.GetTotalFramesDesync();
    state4[3] = d.GetFineTimeOffset();
    fstate3[0] = d.GetSignalAverage();
    fstate3[1] = d.GetCoarseFrequencyOffset();
    fstate3[2] = d.GetFineFrequencyOffset();
}
API void ref_ofdm_reset(void* h) { ((RefOfdm*)h)->demod->Reset(); }
API void ref_ofdm_set_coarse_enabled(void* h, int en) { ((RefOfdm*)h)->demod->GetConfig().sync.is_coarse_freq_correction = en != 0; }
// OFDM_Demod::GetConfig() edited the way the plugin's GUI edits it between Process() calls; f8 / i3 in the order of
// dabgpu_ofdm_config: f8 = {l1 update_beta, thresh_null_start, thresh_null_end, fine_freq_update_beta,
// max_coarse_freq_correction_norm, coarse_freq_slow_beta, impulse_peak_threshold_db, impulse_peak_distance_probability},
// i3 = {l1 nb_samples, l1 nb_decimate, is_coarse_freq_correction}
API void ref_ofdm_set_config(void* h, const float* f8, const int* i3) {
    auto& c = ((RefOfdm*)h)->demod->GetConfig();
    c.signal_l1.update_beta = f8[0];
    c.signal_l1.nb_samples = i3[0];
    c.signal_l1.nb_decimate = i3[1];
    c.null_l1_search.thresh_null_start = f8[1];
    c.null_l1_search.thresh_null_end = f8[2];
    c.sync.fine_freq_update_beta = f8[3];
    c.sync.is_coarse_freq_correction = i3[2] != 0;
    c.sync.max_coarse_freq_correction_norm = f8[4];
    c.sync.coarse_freq_slow_beta = f8[5];
    c.sync.impulse_peak_threshold_db = f8[6];
    c.sync.impulse_peak_distance_probability = f8[7];
}

// Diagnostic taps for stage-level parity (valid after a frame callback, serial driver only)
API void ref_ofdm_get_frame_fft(void* h, float* out, int n_complex) {
    auto s = ((RefOfdm*)h)->demod->GetFrameFFT();
    const size_t n = (size_t(n_complex) < s.size()) ? size_t(n_complex) : s.size();
    memcpy(out, s.data(), n*sizeof(std::complex<float>));
}
API void ref_ofdm_get_frame_data_vec(void* h, float* out, int n_complex) {
    auto s = ((RefOfdm*)h)->demod->GetFrameDataVec();
    const size_t n = (size_t(n_complex) < s.size()) ? size_t(n_complex) : s.size();
    memcpy(out, s.data(), n*sizeof(std::complex<float>));
}
API int ref_ofdm_get_correlation_buffer(void* h, float* out, int n_complex) {
    auto s = ((RefOfdm*)h)->demod->GetCorrelationTimeBuffer();
    const size_t n = (size_t(n_complex) < s.size()) ? size_t(n_complex) : s.size();
    memcpy(out, s.data(), n*sizeof(std::complex<float>));
    return int(n);
}
API void ref_ofdm_get_impulse_response(void* h, float* out, int n) {
    auto s = ((RefOfdm*)h)->demod->GetImpulseResponse();
    const size_t m = (size_t(n) < s.size()) ? size_t(n) : s.size();
    memcpy(out, s.data(), m*sizeof(float));
}
API void ref_ofdm_get_coarse_response(void* h, float* out, int n) {
    auto s = ((RefOfdm*)h)->demod->GetCoarseFrequencyResponse();
    const size_t m = (size_t(n) < s.size()) ? size_t(n) : s.size();
    memcpy(out, s.data(), m*sizeof(float));
}

// ---------------------------------------------------------------------------------------------
// Whole-chain CPU timing helpers (used by bench.py's cpu_baseline / --impl reference leg)
// ---------------------------------------------------------------------------------------------
// Runs OFDM_Demod (free running, threads=1 like the plugin) over a u8 recording in blocks of
// block_size samples, returns seconds of wall time; frames are counted, not stored.
API double ref_time_ofdm_u8(int mode, const uint8_t* iq, long n_samples, int block_size, int repeat, int* frames_out) {
    auto* r = (RefOfdm*)ref_ofdm_create(mode, 1);
    if (!r) return -1.0;
    r->keep_frames = false;
    std::vector<std::complex<float>> buf(static_cast<size_t>(block_size));
    constexpr float BIAS = 127.5f;
    constexpr float scale = 1.0f/127.5f;
    const auto t0 = std::chrono::steady_clock::now();
    for (int rep = 0; rep < repeat; rep++) {
        for (long off = 0; off < n_samples; off += block_size) {
            const long n = (n_samples - off < block_size) ? (n_samples - off) : block_size;
            for (long i = 0; i < n; i++) {
                buf[size_t(i)] = std::complex<float>((float(iq[2*(off+i)]) - BIAS)*scale, (float(iq[2*(off+i)+1]) - BIAS)*scale);
            }
            r->demod->Process({buf.data(), size_t(n)});
        }
    }
    ref_ofdm_flush(r);
    const auto t1 = std::chrono::steady_clock::now();
    if (frames_out) *frames_out = r->demod->GetTotalFramesRead();
    ref_ofdm_destroy(r);
    return std::chrono::duration<double>(t1-t0).count();
}

// Whole receive chain on the CPU, one stream, one thread of control: OFDM_Demod (serial driver, threads=1) -> 4 x
// FIC_Decoder::DecodeFIBGroup + MSC_Decoder::DecodeCIF per sub-channel and CIF + AAC_Frame_Processor::Process for the
// DAB+ sub-channels.  subs = n_subs x {start_address, length, is_uep, uep_index, eep_level, eep_type_b, is_dabplus}.
// counts_out[8] = {frames, fibs_ok, msc_bytes, access_units, superframe headers, RS errors, AU CRC errors, firecode errors} (observer
// events of all sub-channels; bench.py's spot check compares them with the GPU's counters).  Returns seconds of wall time.
// split_out[4] (may be NULL) = seconds spent in {OFDM_Demod::Process incl. the u8 -> float conversion, FIC_Decoder, MSC_Decoder::DecodeCIF,
// AAC_Frame_Processor::Process (fire code, RS(120,110), AU CRCs)}: the per-stage split SURVEY.md section 8(d) asks for.
API double ref_time_chain_split_u8(int mode, const uint8_t* iq, long n_samples, int block_size, int repeat, const int* subs, int n_subs,
                                   long long* counts_out, double* split_out) {
    using clk = std::chrono::steady_clock;
    double t_ofdm = 0, t_fic = 0, t_msc = 0, t_aac = 0;
    auto lap = [](clk::time_point& mark, double& acc) { const auto now = clk::now(); acc += std::chrono::duration<double>(now - mark).count(); mark = now; };
    int dp[13];
    if (ref_dab_params(mode, dp) != 0) return -1.0;
    const DAB_Parameters P = get_dab_parameters(mode);
    auto* r = (RefOfdm*)ref_ofdm_create(mode, 1);
    if (!r) return -1.0;
    r->keep_frames = true;
    void* fic = ref_fic_create(P.nb_fib_cif_bits, P.nb_fibs_per_cif);
    std::vector<void*> msc, aac;
    for (int k = 0; k < n_subs; k++) {
        const int* s = subs + 7*k;
        msc.push_back(ref_msc_create(s[0], s[1], s[2], s[3], s[4], s[5]));
        aac.push_back(s[6] ? ref_aac_create() : nullptr);
    }
    std::vector<int8_t> frame(static_cast<size_t>(P.nb_frame_bits));
    std::vector<uint8_t> bytes(8192), log(1 << 16), fibs(30*8);
    long long frames = 0, fibs_ok = 0, msc_bytes = 0, aus = 0, headers = 0, rs_err = 0, au_crc = 0, fire = 0;
    const auto t0 = std::chrono::steady_clock::now();
    for (int rep = 0; rep < repeat; rep++) {
        for (long off = 0; off < n_samples; off += block_size) {
            const long n = (n_samples - off < block_size) ? (n_samples - off) : block_size;
            auto mark = clk::now();
            ref_ofdm_process_u8(r, iq + 2*off, int(n), 1);
            float cf[2]; int to;
            while (ref_ofdm_pop_frame(r, frame.data(), cf, &to) > 0) {
                lap(mark, t_ofdm);
                frames++;
                if (P.nb_fib_cif_bits == 2304) {
                    for (int c = 0; c < P.nb_cifs; c++) fibs_ok += ref_fic_decode_group(fic, frame.data() + c*P.nb_fib_cif_bits, P.nb_fib_cif_bits, c, fibs.data(), 8);
                }
                lap(mark, t_fic);
                for (int c = 0; c < P.nb_cifs; c++) {
                    const int8_t* cif = frame.data() + P.nb_fic_bits + c*P.nb_cif_bits;
                    for (int k = 0; k < n_subs; k++) {
                        const int nb = ref_msc_decode_cif(msc[size_t(k)], cif, P.nb_cif_bits, bytes.data(), int(bytes.size()));
                        lap(mark, t_msc);
                        if (nb > 0) {
                            msc_bytes += nb;
                            if (aac[size_t(k)]) {
                                auto* a = (RefAac*)aac[size_t(k)];
                                a->log.clear();
                                a->proc.Process({bytes.data(), size_t(nb)});
                                for (size_t o = 0; o + 24 <= a->log.size();) {
                                    int32_t hdr[6];
                                    memcpy(hdr, &a->log[o], 24);
                                    if (hdr[0] == EV_AU) aus++;
                                    else if (hdr[0] == EV_HEADER) headers++;
                                    else if (hdr[0] == EV_RS_ERROR) rs_err++;
                                    else if (hdr[0] == EV_AU_CRC_ERROR) au_crc++;
                                    else if (hdr[0] == EV_FIRECODE_ERROR) fire++;
                                    o += 24 + ((size_t(hdr[5]) + 3u) & ~size_t(3));
                                }
                                lap(mark, t_aac);
                            }
                        }
                    }
                }
            }
            lap(mark, t_ofdm);
        }
    }
    const auto t1 = std::chrono::steady_clock::now();
    if (counts_out) {
        counts_out[0] = frames; counts_out[1] = fibs_ok; counts_out[2] = msc_bytes; counts_out[3] = aus;
        counts_out[4] = headers; counts_out[5] = rs_err; counts_out[6] = au_crc; counts_out[7] = fire;
    }
    if (split_out) { split_out[0] = t_ofdm; split_out[1] = t_fic; split_out[2] = t_msc; split_out[3] = t_aac; }
    for (auto* m : msc) ref_msc_destroy(m);
    for (auto* a : aac) if (a) ref_aac_destroy(a);
    ref_fic_destroy(fic);
    ref_ofdm_destroy(r);
    return std::chrono::duration<double>(t1-t0).count();
}

API double ref_time_chain_u8(int mode, const uint8_t* iq, long n_samples, int block_size, int repeat, const int* subs, int n_subs,
                             long long* counts_out) {
    return ref_time_chain_split_u8(mode, iq, n_samples, block_size, repeat, subs, n_subs, counts_out, nullptr);
}

// ---- FIG processing: FIBs -> the reference's database (SURVEY.md section 8(f) rank 1) --------------------------------
// FIG_Processor (dab/fic/fig_processor.h) -> Radio_FIG_Handler (dab/radio_fig_handler.h) -> DAB_Database_Updater
// (dab/database/dab_database_updater.h), exactly the chain BasicFICRunner builds (basic_radio/basic_fic_runner.cpp:9-32).
#include "dab/fic/fig_processor.h"
#include "dab/radio_fig_handler.h"
#include "dab/dab_misc_info.h"
#include "dab/database/dab_database.h"
#include "dab/database/dab_database_updater.h"

struct RefFig {
    FIG_Processor proc;
    Radio_FIG_Handler handler;
    DAB_Database_Updater updater;
    DAB_Misc_Info misc;
    RefFig() {
        handler.SetUpdater(&updater);
        handler.SetMiscInfo(&misc);
        proc.SetHandler(&handler);
    }
};

API void* ref_fig_create() { return new RefFig(); }
API void ref_fig_destroy(void* p) { delete (RefFig*)p; }
API void ref_fig_process_fib(void* p, const uint8_t* fib30) { ((RefFig*)p)->proc.ProcessFIB({fib30, size_t(30)}); }
// same row formats as dabgpu_autocfg_dump (include/dabgpu.h)
API int ref_fig_dump(void* p, int32_t* subs, int subs_cap, int32_t* comps, int comps_cap, int* n_comps) {
    const auto& db = ((RefFig*)p)->updater.GetDatabase();
    int ns = 0;
    for (const auto& s : db.subchannels) {
        if (ns >= subs_cap) break;
        int32_t* r = subs + ns*9;
        r[0] = s.id; r[1] = s.start_address; r[2] = s.length; r[3] = s.is_uep; r[4] = s.uep_prot_index; r[5] = s.eep_prot_level;
        r[6] = int(uint8_t(s.eep_type)); r[7] = int(uint8_t(s.fec_scheme)); r[8] = s.is_complete;
        ns++;
    }
    int nc = 0;
    for (const auto& c : db.service_components) {
        if (nc >= comps_cap) break;
        int32_t* r = comps + nc*10;
        r[0] = int32_t(c.service_id.value); r[1] = int(uint8_t(c.service_id.type)); r[2] = c.component_id; r[3] = c.subchannel_id; r[4] = c.global_id;
        r[5] = int(uint8_t(c.transport_mode)); r[6] = int(uint8_t(c.audio_service_type)); r[7] = int(uint8_t(c.data_service_type));
        r[8] = c.packet_address; r[9] = c.is_complete;
        nc++;
    }
    *n_comps = nc;
    return ns;
}

// ---- capture file formats of the reference's tools (SURVEY.md section 8(f) rank 3) -----------------------------------
// The reference's own reader chain (examples/app_helpers/app_iq_readers.h:75-159) fed from a memory buffer, and its
// soft-bit <-> hard-byte converters (examples/app_helpers/app_viterbi_convert_block.h:12-44).
#include "app_helpers/app_iq_readers.h"
#include "app_helpers/app_viterbi_convert_block.h"

API long ref_iq_convert(const char* mode, const uint8_t* raw, size_t n_bytes, float* out, size_t out_cap_floats) {
    try {
        FILE* fp = fmemopen(const_cast<uint8_t*>(raw), n_bytes, "rb");   // the reference's InputFile wraps (and closes) a FILE*
        if (!fp) return -1;
        auto file = std::make_shared<InputFile<uint8_t>>(fp);
        auto reader = get_iq_file_reader_from_mode_string(file, mode);
        const size_t n = reader->read({reinterpret_cast<std::complex<float>*>(out), out_cap_floats/2});
        return long(2*n);
    } catch (const std::exception&) {
        return -1;
    }
}
API void ref_softbits_to_bytes(const int8_t* bits, size_t n_bytes, uint8_t* bytes) { convert_viterbi_bits_to_bytes({bits, n_bytes*8}, {bytes, n_bytes}); }
API void ref_bytes_to_softbits(const uint8_t* bytes, size_t n_bytes, int8_t* bits) { convert_viterbi_bytes_to_bits({bytes, n_bytes}, {bits, n_bytes*8}); }
