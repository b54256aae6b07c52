// tests/host/adapter_check.cpp -- drives the C++ adapter classes (host/dab_adapters.hpp) the way the reference's
// own code drives DAB_Viterbi_Decoder / FIC_Decoder / MSC_Decoder / Reed_Solomon_Decoder / AAC_Frame_Processor /
// Radio_Block, on inputs written by tests/test_adapters_gpu.py, and writes what the observers saw.  The Python side
// compares that with the oracle.  Usage: adapter_check <what> <in.bin> <out.bin>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include "../../sdrplusplus-dab-radio-plugin_b200/host/dab_adapters.hpp"

using namespace dabgpu_host;

struct Reader {
    std::vector<uint8_t> buf;
    size_t pos = 0;
    explicit Reader(const char* path) {
        std::ifstream f(path, std::ios::binary);
        buf.assign(std::istreambuf_iterator<char>(f), std::istreambuf_iterator<char>());
    }
    int32_t i32() { int32_t v; memcpy(&v, buf.data() + pos, 4); pos += 4; return v; }
    float f32() { float v; memcpy(&v, buf.data() + pos, 4); pos += 4; return v; }
    const uint8_t* bytes(size_t n) { const uint8_t* p = buf.data() + pos; pos += n; return p; }
};
struct Writer {
    std::vector<uint8_t> buf;
    void i32(int32_t v) { const uint8_t* p = reinterpret_cast<const uint8_t*>(&v); buf.insert(buf.end(), p, p + 4); }
    void u64(uint64_t v) { const uint8_t* p = reinterpret_cast<const uint8_t*>(&v); buf.insert(buf.end(), p, p + 8); }
    void f32(float v) { const uint8_t* p = reinterpret_cast<const uint8_t*>(&v); buf.insert(buf.end(), p, p + 4); }
    void bytes(const void* p, size_t n) { const uint8_t* q = static_cast<const uint8_t*>(p); buf.insert(buf.end(), q, q + n); }
    void save(const char* path) { std::ofstream f(path, std::ios::binary); f.write(reinterpret_cast<const char*>(buf.data()), std::streamsize(buf.size())); }
};

// n_jobs; per job: n_seg, per seg {code_len, code bytes, requested}, n_soft, soft, n_out_bytes
static void run_viterbi(Reader& in, Writer& out) {
    DAB_Viterbi_Decoder dec;
    const int n_jobs = in.i32();
    for (int j = 0; j < n_jobs; j++) {
        const int n_seg = in.i32();
        struct Seg { std::vector<uint8_t> code; int req; };
        std::vector<Seg> segs;
        for (int s = 0; s < n_seg; s++) {
            const int len = in.i32();
            Seg sg;
            const uint8_t* c = in.bytes(size_t(len));
            sg.code.assign(c, c + len);
            sg.req = in.i32();
            segs.push_back(sg);
        }
        const int n_soft = in.i32();
        const int8_t* soft = reinterpret_cast<const int8_t*>(in.bytes(size_t(n_soft)));
        const int n_out = in.i32();
        // the call sequence of FIC_Decoder::DecodeFIBGroup / MSC_Decoder::DecodeEEP
        dec.set_traceback_length(size_t(n_out) * 8);
        dec.reset();
        size_t curr = 0;
        for (const auto& sg : segs)
            curr += dec.update(span<const viterbi_bit_t>(soft + curr, size_t(n_soft) - curr), span<const uint8_t>(sg.code.data(), sg.code.size()), size_t(sg.req));
        std::vector<uint8_t> bytes(static_cast<size_t>(n_out));
        const uint64_t err = dec.chainback(span<uint8_t>(bytes.data(), bytes.size()));
        out.i32(int32_t(curr));
        out.u64(err);
        out.bytes(bytes.data(), bytes.size());
    }
}

static void run_fic(Reader& in, Writer& out) {
    const int n_groups = in.i32();
    FIC_Decoder fic(2304, 3);
    int n_fibs = 0;
    std::vector<uint8_t> fibs;
    fic.OnFIB().Attach([&](span<const uint8_t> fib) { n_fibs++; fibs.insert(fibs.end(), fib.begin(), fib.end()); });
    for (int g = 0; g < n_groups; g++) {
        const int8_t* soft = reinterpret_cast<const int8_t*>(in.bytes(2304));
        n_fibs = 0;
        fibs.clear();
        fic.DecodeFIBGroup(span<const viterbi_bit_t>(soft, 2304), size_t(g % 4));
        out.i32(n_fibs);
        out.bytes(fibs.data(), fibs.size());
    }
}

static Subchannel read_sub(Reader& in, bool* dabplus) {
    Subchannel s;
    s.id = uint8_t(in.i32());
    s.start_address = uint16_t(in.i32());
    s.length = uint16_t(in.i32());
    s.is_uep = in.i32() != 0;
    s.uep_prot_index = uint8_t(in.i32());
    s.eep_prot_level = uint8_t(in.i32());
    s.eep_type = in.i32() ? EEP_Type::TYPE_B : EEP_Type::TYPE_A;
    const int dp = in.i32();
    if (dabplus) *dabplus = dp != 0;
    return s;
}

static void run_msc(Reader& in, Writer& out) {
    const Subchannel s = read_sub(in, nullptr);
    const int n_cifs = in.i32();
    MSC_Decoder dec(s);
    if (!dec.IsValid()) { std::cerr << "MSC_Decoder: " << dec.LastError() << "\n"; exit(2); }
    for (int c = 0; c < n_cifs; c++) {
        const int8_t* cif = reinterpret_cast<const int8_t*>(in.bytes(55296));
        auto bytes = dec.DecodeCIF(span<const viterbi_bit_t>(cif, 55296));
        out.i32(int32_t(bytes.size()));
        out.bytes(bytes.data(), bytes.size());
    }
}

static void run_rs(Reader& in, Writer& out) {
    const int n = in.i32(), nroots = in.i32(), pad = in.i32();
    Reed_Solomon_Decoder rs(8, 0x11D, 0, 1, nroots, pad);
    const int len = 255 - pad;
    for (int i = 0; i < n; i++) {
        const uint8_t* src = in.bytes(size_t(len));
        std::vector<uint8_t> cw(src, src + len);
        std::vector<int> pos(static_cast<size_t>(nroots), 0);
        const int cnt = rs.Decode(cw.data(), pos.data(), 0);
        out.i32(cnt);
        out.bytes(cw.data(), cw.size());
        for (int k = 0; k < nroots; k++) out.i32(k < cnt ? pos[size_t(k)] : 0);
    }
}

// n_bufs; per buffer: len, bytes  ->  per buffer: consumed, n_callbacks, per callback {len, is_corrected, bytes}
static void run_pktfec(Reader& in, Writer& out) {
    MSC_Reed_Solomon_Data_Packet_Processor proc;
    Writer* sink = &out;
    int fired = 0;
    Writer tmp;
    proc.SetCallback([&](span<const uint8_t> pkt, bool corrected) {
        fired++;
        tmp.i32(int32_t(pkt.size())); tmp.i32(corrected ? 1 : 0); tmp.bytes(pkt.data(), pkt.size());
    });
    const int n = in.i32();
    for (int i = 0; i < n; i++) {
        const int len = in.i32();
        const uint8_t* p = in.bytes(size_t(len));
        fired = 0; tmp.buf.clear();
        const size_t used = proc.ReadPacket({p, size_t(len)});
        sink->i32(int32_t(used)); sink->i32(fired); sink->bytes(tmp.buf.data(), tmp.buf.size());
    }
}

struct EventSink {
    Writer& out;
    int n = 0;
    Writer tmp;
    explicit EventSink(Writer& o) : out(o) {}
    void ev(int type, int a, int b, int c, int d, const uint8_t* p, size_t len) {
        n++;
        tmp.i32(type); tmp.i32(a); tmp.i32(b); tmp.i32(c); tmp.i32(d); tmp.i32(int32_t(len));
        tmp.bytes(p, len);
    }
    void attach(DabPlusObservers* o, AAC_Frame_Processor* p) {
        auto fire = [this](const int f, const uint16_t got, const uint16_t calc) { ev(DABGPU_EV_FIRECODE_ERROR, f, got, calc, 0, nullptr, 0); };
        auto rs = [this](const int i, const int t) { ev(DABGPU_EV_RS_ERROR, i, t, 0, 0, nullptr, 0); };
        auto hdr = [this](SuperFrameHeader h) {
            ev(DABGPU_EV_SUPERFRAME_HEADER, int(h.sampling_rate), (h.is_parametric_stereo ? 1 : 0) | (h.is_spectral_band_replication ? 2 : 0) | (h.is_stereo ? 4 : 0),
               int(h.mpeg_surround), 0, nullptr, 0);
        };
        auto crc = [this](const int i, const int t, const uint16_t got, const uint16_t calc) { ev(DABGPU_EV_AU_CRC_ERROR, i, t, got, calc, nullptr, 0); };
        auto au = [this](const int i, const int t, span<uint8_t> b) { ev(DABGPU_EV_ACCESS_UNIT, i, t, 0, 0, b.data(), b.size()); };
        if (o) { o->firecode_error.Attach(fire); o->rs_error.Attach(rs); o->superframe_header.Attach(hdr); o->au_crc_error.Attach(crc); o->access_unit.Attach(au); }
        if (p) { p->OnFirecodeError().Attach(fire); p->OnRSError().Attach(rs); p->OnSuperFrameHeader().Attach(hdr); p->OnAccessUnitCRCError().Attach(crc); p->OnAccessUnit().Attach(au); }
    }
    void flush() { out.i32(n); out.bytes(tmp.buf.data(), tmp.buf.size()); n = 0; tmp.buf.clear(); }
};

static void run_aac(Reader& in, Writer& out) {
    const int n_frames = in.i32(), nbytes = in.i32();
    AAC_Frame_Processor proc;
    EventSink sink(out);
    sink.attach(nullptr, &proc);
    for (int i = 0; i < n_frames; i++) {
        proc.Process(span<const uint8_t>(in.bytes(size_t(nbytes)), size_t(nbytes)));
        sink.flush();
    }
}

// mode, n_subs, subs, block, n_samples, u8 IQ.  Output: stream of records {tag, ...} in observer order.
static void run_radio(Reader& in, Writer& out) {
    const int mode = in.i32(), n_subs = in.i32();
    std::vector<std::pair<Subchannel, bool>> subs;
    for (int i = 0; i < n_subs; i++) { bool dp; const Subchannel s = read_sub(in, &dp); subs.push_back({s, dp}); }
    const int block = in.i32(), n_samples = in.i32();
    const uint8_t* u8 = in.bytes(size_t(n_samples) * 2);
    Radio_Block rb(1, 1, mode);
    auto demod = rb.get_ofdm_demodulator();
    auto radio = rb.get_basic_radio();
    if (!radio->SetSubchannels(subs)) { std::cerr << "SetSubchannels: " << radio->LastError() << "\n"; exit(2); }
    demod->On_OFDM_Frame().Attach([&](span<const viterbi_bit_t> f) { out.i32(1); out.i32(int32_t(f.size())); out.bytes(f.data(), f.size()); out.i32(demod->GetFrameInfo().fine_time_offset); });
    radio->On_FIB().Attach([&](span<const uint8_t> fib) { out.i32(2); out.bytes(fib.data(), 30); });
    for (size_t k = 0; k < subs.size(); k++) {
        radio->Get_Channel(k)->on_msc_data.Attach([&out, k](span<const uint8_t> b) { out.i32(3); out.i32(int32_t(k)); out.i32(int32_t(b.size())); out.bytes(b.data(), b.size()); });
    }
    // QuantisedIQToFloatIQ (examples/app_helpers/app_iq_readers.h:23-43): the plugin interface is complex<float>
    std::vector<std::complex<float>> blockbuf(static_cast<size_t>(block));
    for (int off = 0; off + block <= n_samples; off += block) {
        for (int i = 0; i < block; i++)
            blockbuf[size_t(i)] = std::complex<float>((float(u8[2 * (off + i)]) - 127.5f) * (1.0f / 127.5f), (float(u8[2 * (off + i) + 1]) - 127.5f) * (1.0f / 127.5f));
        demod->Process(span<const std::complex<float>>(blockbuf.data(), blockbuf.size()));
    }
    out.i32(0);
    out.i32(demod->GetTotalFramesRead());
    out.i32(demod->GetTotalFramesDesync());
    out.i32(int(demod->GetState()));
    out.f32(demod->GetNetFrequencyOffset());
}

// mode, n_frames, frame_bits, soft-bit frames.  BasicRadio configures itself from the FIC (EnableSelfConfiguration).
// Output records: {4, id, start, length, is_uep, uep_index, eep_level, eep_type_b, is_dabplus, frame} when a channel is announced,
// {3, id, n, bytes} per decoded logical frame, {0, n_channels} at the end.
static void run_selfcfg(Reader& in, Writer& out) {
    const int mode = in.i32(), n_frames = in.i32(), frame_bits = in.i32();
    BasicRadio radio(get_dab_parameters(mode), 1);
    radio.EnableSelfConfiguration();
    int frame = 0;
    radio.On_Audio_Channel().Attach([&](subchannel_id_t id, BasicRadio::Channel& ch) {
        const Subchannel& s = ch.subchannel;
        out.i32(4); out.i32(id); out.i32(s.start_address); out.i32(s.length); out.i32(s.is_uep); out.i32(s.uep_prot_index); out.i32(s.eep_prot_level);
        out.i32(s.eep_type == EEP_Type::TYPE_B); out.i32(ch.is_dabplus); out.i32(frame);
        ch.on_msc_data.Attach([&out, id](span<const uint8_t> b) { out.i32(3); out.i32(id); out.i32(int32_t(b.size())); out.bytes(b.data(), b.size()); });
    });
    for (frame = 0; frame < n_frames; frame++) {
        const int8_t* f = reinterpret_cast<const int8_t*>(in.bytes(size_t(frame_bits)));
        radio.Process(span<const viterbi_bit_t>(f, size_t(frame_bits)));
    }
    out.i32(0);
    out.i32(int32_t(radio.GetTotalChannels()));
}

// n_decoders, per decoder a sub-channel, n_cifs, then per CIF index one CIF of 55296 soft bits per decoder.  Several MSC_Decoder
// objects alive at once share a pool context (host/dab_adapters.hpp MscPool), one leased stream each; a decoder destroyed and
// re-created in between must start with an empty de-interleaver.
static void run_mscpool(Reader& in, Writer& out) {
    const int n_dec = in.i32();
    std::vector<Subchannel> subs;
    for (int i = 0; i < n_dec; i++) subs.push_back(read_sub(in, nullptr));
    const int n_cifs = in.i32();
    { MSC_Decoder scratch(subs[0]); const std::vector<int8_t> z(55296, 0); scratch.DecodeCIF(span<const viterbi_bit_t>(z.data(), z.size())); }   // leases and returns stream 0
    std::vector<std::unique_ptr<MSC_Decoder>> dec;
    for (int i = 0; i < n_dec; i++) {
        dec.push_back(std::make_unique<MSC_Decoder>(subs[size_t(i)]));
        if (!dec.back()->IsValid()) { std::cerr << "MSC_Decoder: " << dec.back()->LastError() << "\n"; exit(2); }
    }
    for (int c = 0; c < n_cifs; c++)
        for (int i = 0; i < n_dec; i++) {
            const int8_t* cif = reinterpret_cast<const int8_t*>(in.bytes(55296));
            auto bytes = dec[size_t(i)]->DecodeCIF(span<const viterbi_bit_t>(cif, 55296));
            out.i32(int32_t(bytes.size()));
            out.bytes(bytes.data(), bytes.size());
        }
}

// mode, block, n_samples, u8 IQ through Create_OFDM_Demodulator; then the GUI getters of OFDM_Demod (ofdm_demodulator.h:135-139,
// polled by src/render_radio_block.cpp:96-214): sizes and contents as floats.
static void run_taps(Reader& in, Writer& out) {
    const int mode = in.i32(), block = in.i32(), n_samples = in.i32();
    const uint8_t* u8 = in.bytes(size_t(n_samples) * 2);
    auto demod = Create_OFDM_Demodulator(mode, 1);
    std::vector<std::complex<float>> blockbuf(static_cast<size_t>(block));
    for (int off = 0; off + block <= n_samples; off += block) {
        for (int i = 0; i < block; i++)
            blockbuf[size_t(i)] = std::complex<float>((float(u8[2 * (off + i)]) - 127.5f) * (1.0f / 127.5f), (float(u8[2 * (off + i) + 1]) - 127.5f) * (1.0f / 127.5f));
        demod->Process(span<const std::complex<float>>(blockbuf.data(), blockbuf.size()));
    }
    out.i32(demod->GetTotalFramesRead());
    const auto imp = demod->GetImpulseResponse();
    out.i32(int32_t(imp.size())); out.bytes(imp.data(), imp.size() * sizeof(float));
    const auto coarse = demod->GetCoarseFrequencyResponse();
    out.i32(int32_t(coarse.size())); out.bytes(coarse.data(), coarse.size() * sizeof(float));
    const auto fft = demod->GetFrameFFT();
    out.i32(int32_t(fft.size())); out.bytes(fft.data(), fft.size() * sizeof(std::complex<float>));
    const auto vec = demod->GetFrameDataVec();
    out.i32(int32_t(vec.size())); out.bytes(vec.data(), vec.size() * sizeof(std::complex<float>));
    const auto corr = demod->GetCorrelationTimeBuffer();
    out.i32(int32_t(corr.size())); out.bytes(corr.data(), corr.size() * sizeof(std::complex<float>));
}

// mode, n_edits, per edit {call index, 8 floats, 3 ints} (the fields of dabgpu_ofdm_config, floats and ints each in its order),
// n_calls, call lengths, u8 IQ.  Each call is one OFDM_Demod::Process block; before the calls that have an edit, every field of
// OFDM_Demod::GetConfig() is written the way the plugin's GUI writes it.  Output per call: n_frames, per frame {bits, coarse, fine,
// fine time offset}, then GetState, GetTotalFramesRead, GetTotalFramesDesync, GetFineTimeOffset, GetSignalAverage,
// GetCoarseFrequencyOffset, GetFineFrequencyOffset.
static void run_ofdmcfg(Reader& in, Writer& out) {
    const int mode = in.i32(), n_edits = in.i32();
    struct Edit { int call; float f[8]; int i[3]; };
    std::vector<Edit> edits(static_cast<size_t>(n_edits));
    for (auto& e : edits) {
        e.call = in.i32();
        for (float& v : e.f) v = in.f32();
        for (int& v : e.i) v = in.i32();
    }
    const int n_calls = in.i32();
    std::vector<int> lens(static_cast<size_t>(n_calls));
    for (int& l : lens) l = in.i32();
    auto demod = Create_OFDM_Demodulator(mode, 1);
    Writer frames;
    int n_frames = 0;
    demod->On_OFDM_Frame().Attach([&](span<const viterbi_bit_t> f) {
        n_frames++;
        frames.bytes(f.data(), f.size());
        const dabgpu_frame_info& fi = demod->GetFrameInfo();
        frames.f32(fi.freq_coarse_offset); frames.f32(fi.freq_fine_offset); frames.i32(fi.fine_time_offset);
    });
    std::vector<std::complex<float>> blockbuf;
    for (int k = 0; k < n_calls; k++) {
        for (const auto& e : edits) {
            if (e.call != k) continue;
            auto& c = demod->GetConfig();
            c.signal_l1.update_beta = e.f[0];
            c.signal_l1.nb_samples = e.i[0];
            c.signal_l1.nb_decimate = e.i[1];
            c.null_l1_search.thresh_null_start = e.f[1];
            c.null_l1_search.thresh_null_end = e.f[2];
            c.sync.fine_freq_update_beta = e.f[3];
            c.sync.is_coarse_freq_correction = e.i[2] != 0;
            c.sync.max_coarse_freq_correction_norm = e.f[4];
            c.sync.coarse_freq_slow_beta = e.f[5];
            c.sync.impulse_peak_threshold_db = e.f[6];
            c.sync.impulse_peak_distance_probability = e.f[7];
        }
        const int n = lens[size_t(k)];
        const uint8_t* u8 = in.bytes(size_t(n) * 2);
        blockbuf.resize(size_t(n));
        for (int i = 0; i < n; i++)
            blockbuf[size_t(i)] = std::complex<float>((float(u8[2 * i]) - 127.5f) * (1.0f / 127.5f), (float(u8[2 * i + 1]) - 127.5f) * (1.0f / 127.5f));
        n_frames = 0;
        frames.buf.clear();
        demod->Process(span<const std::complex<float>>(blockbuf.data(), blockbuf.size()));
        out.i32(n_frames);
        out.bytes(frames.buf.data(), frames.buf.size());
        out.i32(int(demod->GetState())); out.i32(demod->GetTotalFramesRead()); out.i32(demod->GetTotalFramesDesync());
        out.i32(demod->GetFineTimeOffset());
        out.f32(demod->GetSignalAverage()); out.f32(demod->GetCoarseFrequencyOffset()); out.f32(demod->GetFineFrequencyOffset());
    }
}

int main(int argc, char** argv) {
    if (argc != 4) { std::cerr << "usage: adapter_check <viterbi|fic|msc|mscpool|rs|pktfec|aac|radio|selfcfg|taps|ofdmcfg> in.bin out.bin\n"; return 1; }
    try {
        Reader in(argv[2]);
        Writer out;
        const std::string what = argv[1];
        if (what == "viterbi") run_viterbi(in, out);
        else if (what == "fic") run_fic(in, out);
        else if (what == "msc") run_msc(in, out);
        else if (what == "rs") run_rs(in, out);
        else if (what == "aac") run_aac(in, out);
        else if (what == "pktfec") run_pktfec(in, out);
        else if (what == "radio") run_radio(in, out);
        else if (what == "selfcfg") run_selfcfg(in, out);
        else if (what == "mscpool") run_mscpool(in, out);
        else if (what == "taps") run_taps(in, out);
        else if (what == "ofdmcfg") run_ofdmcfg(in, out);
        else { std::cerr << "unknown test " << what << "\n"; return 1; }
        out.save(argv[3]);
    } catch (const std::exception& e) {
        std::cerr << "adapter_check: " << e.what() << "\n";
        return 3;
    }
    return 0;
}
