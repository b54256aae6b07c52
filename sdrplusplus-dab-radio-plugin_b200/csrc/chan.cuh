// chan.cuh -- channel decoding of whole transmission frames taken from the soft-bit frame ring:
// FIC FIB groups and MSC sub-channels are turned into Viterbi jobs on the device.
//   BasicRadio::Process split            basic_radio/basic_radio.cpp:41-65
//   BasicFICRunner::Process              basic_radio/basic_fic_runner.cpp:34-49
//   FIC_Decoder::DecodeFIBGroup          dab/fic/fic_decoder.cpp:53-117
//   MSC_Decoder::DecodeCIF               dab/msc/msc_decoder.cpp:46-154
//   CIF_Deinterleaver                    dab/msc/cif_deinterleaver.cpp:20-71  (fused into the Viterbi loader as a gather)
#pragma once
#include "viterbi.cuh"
#include "viterbi_lanes.cuh"

#define CIF_OUT_STRIDE 6912u     // decoded bytes per CIF can never exceed 55296/8
#define FIC_GROUP_BYTES 128u     // 96 used in modes I/II/IV

struct SubCfgDev {
    uint32_t start_bit, nb_bits;
    uint32_t seg_step_end[DABGPU_MAX_SEGMENTS];
    uint32_t seg_in_base[DABGPU_MAX_SEGMENTS];
    uint8_t seg_pi[8];
    uint32_t n_seg, total_steps, n_out_bytes, out_offset;
    uint32_t is_dabplus, payload, pad1, pad2;   // payload: DABGPU_PAYLOAD_*
};

struct ChanDev {
    // geometry
    GatherGeom geom;
    uint32_t nb_fibs_per_cif, fib_group_bits, fic_enabled;
    uint32_t max_subs, jobs_per_stream;
    // per-stream state / config
    const int8_t* frames;            // [stream][slot][frame_bits]
    size_t stream_frames_stride;     // slots*frame_bits
    const uint32_t* frames_written;  // [stream] SNAPSHOT of the OFDM stage's counter, taken on the main stream before the channel
                                     // stream forks: the next OFDM stage advances the live counter while this decode runs
    uint32_t* frames_decoded;        // [stream]
    uint32_t max_lag;                // frames_written - frames_decoded above this: the history of the oldest frame is overwritten
    const SubCfgDev* subcfg;         // [stream][max_subs]
    const uint32_t* n_subs;          // [stream]
    uint32_t* cifs_consumed;         // [stream][max_subs]
    // outputs of the last decode
    uint8_t* fic_out;                // [stream][nb_cifs][FIC_GROUP_BYTES]
    uint8_t* fic_crc;                // [stream][nb_cifs][4]
    uint8_t* msc_out;                // [stream][nb_cifs][CIF_OUT_STRIDE]
    uint8_t* msc_valid;              // [stream][nb_cifs][max_subs]
    int8_t* deint;                   // [stream][nb_cifs][cif_bits]: the CIFs of the frame being decoded after the time de-interleaver
    int32_t* status;                 // [stream][2] = {decoded, frame_index}
    unsigned long long* counters;    // see CNT_* below
};

enum { CNT_FRAMES_DEMOD = 0, CNT_FRAMES_CHAN, CNT_FIB_OK, CNT_FIB_TOTAL, CNT_MSC_BYTES, CNT_SF_OK, CNT_SF_RS_FAIL,
       CNT_SF_FIRE_FAIL, CNT_AU_OK, CNT_AU_CRC_FAIL, CNT_FRAMES_DROPPED, CNT_COUNT };

// The frame the channel decoder takes next.  Normally the oldest undecoded one.  When the decoder fell so far behind the OFDM
// stage that the ring slots holding the 16-CIF history of that frame were overwritten (frames_written - frames_decoded >
// max_lag), it skips to the newest frame and restarts every time de-interleaver of the stream empty, like a fresh
// CIF_Deinterleaver (cif_deinterleaver.cpp:38-41): stale soft bits are never decoded as valid.  The reference cannot get there
// (its ThreadedRingBuffer blocks the producer, src/radio_block.cpp:20-44); dropped frames are counted (CNT_FRAMES_DROPPED).
struct ChanPick { uint32_t t; bool has_frame, skipped; };
__device__ __forceinline__ ChanPick chan_pick_frame(const ChanDev& C, const uint32_t s) {
    ChanPick p;
    const uint32_t w = C.frames_written[s], d = C.frames_decoded[s];
    p.has_frame = w > d;
    p.skipped = p.has_frame && (w - d) > C.max_lag;
    p.t = p.skipped ? w - 1u : d;
    return p;
}

// One thread per potential job: (stream, j).  j < nb_cifs => FIB group j; otherwise sub-channel x CIF.
// count_plan (optional): the histogram of trellis lengths that k_vit_plan needs is taken here, where the lengths are at hand,
// instead of by a separate pass over the job array (k_vit_count).
__global__ void k_chan_build_jobs(const ChanDev C, VitJobDev* __restrict__ jobs, const int first_stream, const int n_streams, VlPlan* __restrict__ count_plan) {
    const uint32_t gid = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t total = uint32_t(n_streams) * C.jobs_per_stream;
    const bool in_range = gid < total;            // no early return: the histogram below is taken by whole warps
    const uint32_t si = in_range ? gid / C.jobs_per_stream : 0u, j = in_range ? gid - si * C.jobs_per_stream : 0u;
    const uint32_t s = uint32_t(first_stream) + si;
    VitJobDev J;
    memset(&J, 0, sizeof(J));
    const ChanPick pick = chan_pick_frame(C, s);
    const uint32_t t = pick.t;
    const bool has_frame = pick.has_frame && in_range;
    const uint32_t nb_cifs = C.geom.nb_cifs;
    if (j == 0 && in_range) {
        C.status[2 * s + 0] = has_frame ? 1 : 0;
        C.status[2 * s + 1] = int32_t(t);
    }
    if (has_frame) {
        const int8_t* ring = C.frames + size_t(s) * C.stream_frames_stride;
        if (j < nb_cifs) {
            if (C.fic_enabled) {
                // PI_16 x 21 blocks, PI_15 x 3 blocks, tail (fic_decoder.cpp:74-85)
                J.src = ring + size_t(t & C.geom.slot_mask) * C.geom.frame_bits + size_t(j) * C.fib_group_bits;
                J.out = C.fic_out + (size_t(s) * nb_cifs + j) * FIC_GROUP_BYTES;
                J.crc_ok = C.fic_crc + (size_t(s) * nb_cifs + j) * 4u;
                J.seg_pi[0] = 16; J.seg_pi[1] = 15; J.seg_pi[2] = 0;
                J.seg_step_end[0] = 672; J.seg_step_end[1] = 768; J.seg_step_end[2] = 774;
                J.seg_step_end[3] = 774; J.seg_step_end[4] = 774;
                J.seg_in_base[0] = 0; J.seg_in_base[1] = 2016; J.seg_in_base[2] = 2292;
                J.n_seg = 3; J.total_steps = 774; J.n_out_bytes = 96;
                J.flags = VJ_DESCRAMBLE | VJ_FIB_CRC;
                J.n_fibs = C.nb_fibs_per_cif;
            }
        } else {
            const uint32_t jj = j - nb_cifs;
            const uint32_t sub = jj / nb_cifs, c = jj - sub * nb_cifs;
            if (sub < C.n_subs[s]) {
                const SubCfgDev cfg = C.subcfg[size_t(s) * C.max_subs + sub];
                // CIF_Deinterleaver::Deinterleave returns false until 16 CIFs were consumed (cif_deinterleaver.cpp:38-41)
                const uint32_t consumed = (pick.skipped ? 0u : C.cifs_consumed[size_t(s) * C.max_subs + sub]) + c + 1u;
                const bool valid = consumed >= 16u && cfg.total_steps != 0u;   // total_steps 0: entry removed (dabgpu_msc_remove_subchannel)
                C.msc_valid[(size_t(s) * nb_cifs + c) * C.max_subs + sub] = valid ? 1 : 0;
                if (valid) {
                    // the sub-channel's logical frame, already de-interleaved by k_chan_deinterleave: an ordinary linear job
                    J.src = C.deint + (size_t(s) * nb_cifs + c) * C.geom.cif_bits + cfg.start_bit;
                    J.out = C.msc_out + (size_t(s) * nb_cifs + c) * CIF_OUT_STRIDE + cfg.out_offset;
#pragma unroll
                    for (int i = 0; i < DABGPU_MAX_SEGMENTS; i++) { J.seg_step_end[i] = cfg.seg_step_end[i]; J.seg_in_base[i] = cfg.seg_in_base[i]; }
#pragma unroll
                    for (int i = 0; i < 8; i++) J.seg_pi[i] = cfg.seg_pi[i];
                    J.n_seg = cfg.n_seg; J.total_steps = cfg.total_steps; J.n_out_bytes = cfg.n_out_bytes;
                    J.flags = VJ_DESCRAMBLE;
                }
            }
        }
    }
    if (in_range) jobs[gid] = J;
    if (count_plan != nullptr) vl_count_warp(count_plan, J.total_steps);
}

// CIF_Deinterleaver::Deinterleave (dab/msc/cif_deinterleaver.cpp:20-71) for the nb_cifs CIFs of the frame every stream decodes in
// this call.  Sub-channels start at multiples of 64 bits, so the rule "bit i of a logical frame comes from the CIF that is
// 15 - bitrev4(i mod 16) CIFs old" acts on the whole 55296-bit CIF alike, whatever the sub-channel layout: the kernel writes the
// de-interleaved CIF in natural order and every MSC Viterbi job becomes a linear job over a piece of it.
// One thread per capacity unit (64 soft bits = 4 bytes of each of the 16 planes of the ring layout, viterbi.cuh): 16 word loads,
// each coalesced across the threads of a warp (128 contiguous bytes of one plane), 4x4 byte transposes in registers (32 PRMT),
// four 16-byte stores that are contiguous across the warp as well.  grid = (ceil(cu / blockDim), streams * nb_cifs).
__device__ __forceinline__ void deint_transpose4(const uint32_t a, const uint32_t b, const uint32_t c, const uint32_t d, uint32_t (&o)[4]) {
    const uint32_t t0 = __byte_perm(a, b, 0x5140), t1 = __byte_perm(a, b, 0x7362);
    const uint32_t t2 = __byte_perm(c, d, 0x5140), t3 = __byte_perm(c, d, 0x7362);
    o[0] = __byte_perm(t0, t2, 0x5410); o[1] = __byte_perm(t0, t2, 0x7632);
    o[2] = __byte_perm(t1, t3, 0x5410); o[3] = __byte_perm(t1, t3, 0x7632);
}
__global__ void __launch_bounds__(288) k_chan_deinterleave(const ChanDev C, const int first_stream) {
    const uint32_t nb_cifs = C.geom.nb_cifs;
    const uint32_t si = blockIdx.y / nb_cifs, c = blockIdx.y - si * nb_cifs;
    const uint32_t s = uint32_t(first_stream) + si;
    if (!C.status[2 * s] || C.n_subs[s] == 0u) return;
    const uint32_t cu = blockIdx.x * blockDim.x + threadIdx.x;
    if (cu >= C.geom.cif_bits / 64u) return;
    const uint32_t newest = uint32_t(C.status[2 * s + 1]) * nb_cifs + c;
    const int8_t* ring = C.frames + size_t(s) * C.stream_frames_stride;
    uint32_t p[16];
#pragma unroll
    for (uint32_t r = 0; r < 16u; r++) p[r] = __ldg(reinterpret_cast<const uint32_t*>(ring + (size_t(vit_plane_offset(newest, 0u, C.geom, r)) + 4u * cu)));
    // o[m][kk] = planes 4m..4m+3 at plane byte 4cu + kk = soft bits 64cu + 16kk + 4m .. + 3 of the logical CIF
    uint32_t o[4][4];
#pragma unroll
    for (uint32_t m = 0; m < 4u; m++) deint_transpose4(p[4u * m], p[4u * m + 1u], p[4u * m + 2u], p[4u * m + 3u], o[m]);
    uint4* dst = reinterpret_cast<uint4*>(C.deint + (size_t(s) * nb_cifs + c) * C.geom.cif_bits + 64u * cu);
#pragma unroll
    for (uint32_t kk = 0; kk < 4u; kk++) dst[kk] = make_uint4(o[0][kk], o[1][kk], o[2][kk], o[3][kk]);
}

// One warp per stream: advance the consumption counters after the Viterbi pass (lanes over the sub-channels).
__global__ void __launch_bounds__(32) k_chan_finish(const ChanDev C, const int first_stream, const int n_streams) {
    const uint32_t si = blockIdx.x, lane = threadIdx.x;
    if (si >= uint32_t(n_streams)) return;
    const uint32_t s = uint32_t(first_stream) + si;
    if (!C.status[2 * s]) return;
    const ChanPick pick = chan_pick_frame(C, s);   // same inputs as in k_chan_build_jobs: frames_decoded only changes below
    const uint32_t nb_cifs = C.geom.nb_cifs;
    unsigned long long bytes = 0;
    const uint32_t ns = C.n_subs[s];
    for (uint32_t sub = lane; sub < ns; sub += 32u) {
        uint32_t& cc = C.cifs_consumed[size_t(s) * C.max_subs + sub];
        const uint32_t nb = C.subcfg[size_t(s) * C.max_subs + sub].n_out_bytes;
        for (uint32_t c = 0; c < nb_cifs; c++)
            if (C.msc_valid[(size_t(s) * nb_cifs + c) * C.max_subs + sub]) bytes += nb;
        cc = min((pick.skipped ? 0u : cc) + nb_cifs, 1u << 30);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) bytes += __shfl_xor_sync(FULL_MASK, bytes, o);
    if (lane == 0) {
        if (C.fic_enabled) {
            unsigned long long fib_ok = 0;
            for (uint32_t c = 0; c < nb_cifs; c++)
                for (uint32_t f = 0; f < C.nb_fibs_per_cif; f++) fib_ok += C.fic_crc[(size_t(s) * nb_cifs + c) * 4u + f];
            atomicAdd(&C.counters[CNT_FIB_TOTAL], (unsigned long long)(nb_cifs * C.nb_fibs_per_cif));
            atomicAdd(&C.counters[CNT_FIB_OK], fib_ok);
        }
        atomicAdd(&C.counters[CNT_MSC_BYTES], bytes);
        atomicAdd(&C.counters[CNT_FRAMES_CHAN], 1ull);
        if (pick.skipped) atomicAdd(&C.counters[CNT_FRAMES_DROPPED], (unsigned long long)(pick.t - C.frames_decoded[s]));
        C.frames_decoded[s] = pick.t + 1u;
    }
}
