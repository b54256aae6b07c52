// packet.cuh -- packet-mode data sub-channels inside the channel decode.
//   basic_data_packet_channel.cpp:49-88                       the walk of a logical frame: pos += ReadPacket(frame[pos:])
//   MSC_Reed_Solomon_Data_Packet_Processor::ReadPacket       msc_reed_solomon_data_packet_processor.cpp:49-258 (FEC scheme 1,
//       ETSI EN 300 401 5.3.5: a 2472-byte ring of whole packets, nine FEC packets with counters 0..8 close a set, RS(204,188)
//       over the 12 rows of the 204-column table, only the application data table is corrected)
//   packet CRC                                               EN 300 401 5.3.2 (CRC16-CCITT, the FIB CRC)
//
// One warp per (stream, packet entry).  The entries are a compact list rebuilt when the sub-channel tables change, so a decode
// without packet entries launches nothing.  Each entry owns a region of the packet pool, allocated when it is declared:
//   [PktHdr][ring of PKT_RING bytes][log of pkt_item_bound bytes]
// The log holds the entry's records of the last decode in their final form (dabgpu_event_header + whole packet), so the
// per-sub getter copies it as is and k_packet_pack moves it into the packed output.
#pragma once
#include "dabplus.cuh"
#include <algorithm>
#include <climits>
#include <map>

#define PKT_RING 2472   // 2256 bytes of application data + 9 FEC packets
#define PKT_WARPS 4
#define PKT_HDR_BYTES 32
#define PKT_RING_BYTES 2480   // PKT_RING rounded up to 16
#define PKT_LOG_OFF (PKT_HDR_BYTES + PKT_RING_BYTES)
static_assert(PKT_RING == PKT_FEC_DATA * PKT_FEC_ROWS + 9 * 24, "the ring holds one application data table and its nine FEC packets");

// last = -1: no FEC packet of the current set seen yet (the reference's "no previous counter")
struct PktHdr { int32_t rd, wr, fill, last, log_len, log_cap, pad0, pad1; };
static_assert(sizeof(PktHdr) == PKT_HDR_BYTES, "region header size");
struct PktItemDev { uint32_t stream, sub; uint64_t region; };

// Bound of one packet entry's log per channel decode.  A = nb_cifs x bytes per CIF arrive.  Every packet that leaves was in the
// ring before the decode (at most PKT_RING bytes) or arrived during it, so at most PKT_RING + A bytes of packets leave, in
// records of at least 24 bytes: at most (PKT_RING + A) / 24 PACKET headers.  A set ends only on an FEC packet, which takes 24 bytes
// of the input: at most A / 24 PACKET_FEC records; one more is allowed for.  Packet lengths are multiples of 24, so no record
// carries padding and every record starts 8-byte aligned.
#define PKT_MIN_PACKET 24
static_assert(PKT_MIN_PACKET == 24 && sizeof(dabgpu_event_header) == 24, "records of at least 24 bytes each add a 24-byte header");
static inline uint64_t pkt_item_bound(const uint32_t nb_cifs, const uint32_t n_out_bytes) {
    const uint64_t A = uint64_t(nb_cifs) * n_out_bytes;
    const uint64_t packets = (PKT_RING + A) / PKT_MIN_PACKET;
    return (packets * 24u + (PKT_RING + A) + (A / PKT_MIN_PACKET + 1u) * 24u + 7u) & ~uint64_t(7);
}
static inline uint64_t pkt_region_bytes(const uint64_t log_cap) { return (PKT_LOG_OFF + log_cap + 15u) & ~uint64_t(15); }

struct PktShared : DpTables {
    __align__(16) uint8_t ring[PKT_WARPS][PKT_RING_BYTES];
    __align__(16) uint8_t fec[PKT_WARPS][PKT_FEC_FRAME_BYTES];
    __align__(16) uint8_t pkt[PKT_WARPS][96];
};

// One record into the item's log: the header by lanes 0-5, then n payload bytes from shared memory (n a multiple of 4).  Records
// that would not fit the log are dropped (the bound above says none does).
__device__ __forceinline__ void pkt_record(uint8_t* log, int& off, const int cap, const int type, const int a, const int b, const int c,
                                           const int d, const uint8_t* payload, const int n, const uint32_t lane) {
    if (off + 24 + n > cap) return;
    int32_t* h = reinterpret_cast<int32_t*>(log + off);
    const int v[6] = {type, a, b, c, d, n};
    if (lane < 6u) h[lane] = v[lane];
    uint32_t* dst = reinterpret_cast<uint32_t*>(log + off + 24);
    const uint32_t* src = reinterpret_cast<const uint32_t*>(payload);
    for (int i = int(lane); i < n / 4; i += 32) dst[i] = src[i];
    off += 24 + n;
}

// One packet (staged in shared memory) out through the callback: is_corrected, crc_ok, address.
__device__ __forceinline__ void pkt_deliver(const PktShared& sh, const uint8_t* p, const int n, const int corrected, uint8_t* log, int& off,
                                            const int cap, const uint32_t lane) {
    const uint16_t pred = crc16_ccitt_warp(sh.crc_ccitt, p, n - 2, lane);
    const uint16_t rx = uint16_t((uint16_t(p[n - 2]) << 8) | p[n - 1]);
    pkt_record(log, off, cap, DABGPU_EV_PACKET, corrected, rx == pred ? 1 : 0, ((p[0] & 3) << 8) | p[1], 0, p, n, lane);
    __syncwarp();
}

struct PktRing { int rd, wr, fill, last; };

// Pops every packet of the ring (corrected = 0), or packets while fewer than `limit` bytes left (the corrected release).
__device__ void pkt_release(const PktShared& sh, const uint8_t* ring, uint8_t* pkt, PktRing& R, const int limit, const int corrected, uint8_t* log,
                            int& off, const int cap, const uint32_t lane) {
    int total = 0;
    while (total < limit && R.fill > 0) {
        const int n = 24 * ((ring[R.rd] >> 6) + 1);
        for (int i = int(lane); i < n; i += 32) pkt[i] = ring[(R.rd + i) % PKT_RING];
        __syncwarp();
        pkt_deliver(sh, pkt, n, corrected, log, off, cap, lane);
        R.fill -= n;
        R.rd = (R.rd + n) % PKT_RING;
        total += n;
    }
}

// PerformReedSolomonCorrection on a full ring: the FEC frame is staged in shared memory in the order the adapter builds it
// ([2256 application data | 192 RS data]), lanes 0-11 decode one row each, the application data table goes back into the ring.
// Returns {rows decoded, rows uncorrectable, sum of the decoded rows' error counts} in every lane.  Kept out of line: inlined, the
// RS decoder's registers spill in the walk around it, which runs on every packet while this runs once per 2472 bytes.
__device__ __noinline__ int3 pkt_correct(const PktShared& sh, uint8_t* ring, uint8_t* fec, const PktRing& R, const uint32_t lane) {
    for (int k = int(lane); k < PKT_FEC_FRAME_BYTES; k += 32) {
        int src = k;
        if (k >= PKT_FEC_ROWS * PKT_FEC_DATA) {
            const int i = (k - PKT_FEC_ROWS * PKT_FEC_DATA) / 22, j = (k - PKT_FEC_ROWS * PKT_FEC_DATA) - 22 * i;
            src = PKT_FEC_ROWS * PKT_FEC_DATA + 24 * i + 2 + j;
        }
        fec[k] = ring[(R.rd + src) % PKT_RING];
    }
    __syncwarp();
    int cnt = 0;
    if (lane < uint32_t(PKT_FEC_ROWS)) cnt = pkt_fec_row(GfTables{sh.gf_ex, sh.gf_lg}, fec + lane);
    __syncwarp();
    for (int k = int(lane); k < PKT_FEC_ROWS * PKT_FEC_DATA; k += 32) ring[(R.rd + k) % PKT_RING] = fec[k];
    __syncwarp();
    const bool row = lane < uint32_t(PKT_FEC_ROWS);
    int sum = (row && cnt >= 0) ? cnt : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(FULL_MASK, sum, o);
    return make_int3(__popc(__ballot_sync(FULL_MASK, row && cnt >= 0)), __popc(__ballot_sync(FULL_MASK, row && cnt < 0)), sum);
}

// One logical frame of n bytes walked as basic_data_packet_channel.cpp:49-88 does; every lane keeps the same copy of R.
__device__ void pkt_frame(const PktShared& sh, uint8_t* ring, uint8_t* fec, uint8_t* pkt, const uint8_t* __restrict__ frame, const int n,
                          const bool use_fec, PktRing& R, uint8_t* log, int& off, const int cap, const uint32_t lane) {
    int pos = 0;
    while (n - pos >= 2) {
        const uint8_t b0 = frame[pos], b1 = frame[pos + 1];
        const int counter = (b0 >> 2) & 0xF, address = ((b0 & 3) << 8) | b1;
        const bool is_fec = use_fec && address == 0x3FE;
        const int lid = is_fec ? 0 : (b0 >> 6), len = 24 * (lid + 1);
        if (n - pos < len) break;
        if (!use_fec) {
            for (int i = int(lane); i < len; i += 32) pkt[i] = frame[pos + i];
            __syncwarp();
            pkt_deliver(sh, pkt, len, 0, log, off, cap, lane);
            pos += len;
            continue;
        }
        // push (msc_reed_solomon_data_packet_processor.cpp:137-153): evict the oldest packets until it fits, the stored length id is
        // the one the processor decided on
        while (PKT_RING - R.fill < len) {
            const int m = 24 * ((ring[R.rd] >> 6) + 1);
            R.fill -= m;
            R.rd = (R.rd + m) % PKT_RING;
        }
        for (int i = int(lane); i < len; i += 32) ring[(R.wr + i) % PKT_RING] = frame[pos + i];
        __syncwarp();
        if (lane == 0) ring[R.wr] = uint8_t((b0 & 0x3F) | (lid << 6));
        __syncwarp();
        R.fill += len;
        R.wr = (R.wr + len) % PKT_RING;
        pos += len;
        if (!is_fec) continue;
        const bool invalid = (R.last >= 0) ? (counter != R.last + 1) : (counter != 0);
        if (invalid) {
            R.last = -1;
            pkt_record(log, off, cap, DABGPU_EV_PACKET_FEC, 0, 0, 0, 0, nullptr, 0, lane);
            pkt_release(sh, ring, pkt, R, INT_MAX, 0, log, off, cap, lane);
            continue;
        }
        R.last = counter;
        if (counter != 8) continue;
        if (R.fill != PKT_RING) {
            pkt_record(log, off, cap, DABGPU_EV_PACKET_FEC, 0, 0, 0, 0, nullptr, 0, lane);
            pkt_release(sh, ring, pkt, R, INT_MAX, 0, log, off, cap, lane);
        } else {
            const int3 r = pkt_correct(sh, ring, fec, R, lane);
            pkt_record(log, off, cap, DABGPU_EV_PACKET_FEC, 1, r.x, r.y, r.z, nullptr, 0, lane);
            pkt_release(sh, ring, pkt, R, PKT_FEC_ROWS * PKT_FEC_DATA, 1, log, off, cap, lane);
        }
        R.last = -1;
        R.rd = R.wr = R.fill = 0;
    }
}

// One (stream, packet entry) item: the logical frames the decoder emitted for it (msc_valid), in order.  The log of a stream
// the call did not decode is empty, like a DAB+ entry's.
__device__ void pkt_work_item(PktShared& sh, const ChanDev& C, uint8_t* pool, const PktItemDev it, const uint32_t lane) {
    const uint32_t w = (threadIdx.x >> 5) % PKT_WARPS;
    uint8_t* region = pool + it.region;
    PktHdr* H = reinterpret_cast<PktHdr*>(region);
    const uint32_t s = it.stream, sub = it.sub;
    if (!C.status[2 * s] || sub >= C.n_subs[s]) {
        if (lane == 0) H->log_len = 0;
        return;
    }
    const size_t idx = size_t(s) * C.max_subs + sub;
    const SubCfgDev cfg = C.subcfg[idx];
    const bool use_fec = cfg.payload == DABGPU_PAYLOAD_PACKET_FEC;
    PktRing R{H->rd, H->wr, H->fill, H->last};
    const int cap = H->log_cap;
    uint8_t* ring = sh.ring[w];
    uint8_t* ring_g = region + PKT_HDR_BYTES;
    if (use_fec && R.fill > 0) {
        for (int i = int(lane); i < PKT_RING_BYTES / 16; i += 32) reinterpret_cast<uint4*>(ring)[i] = reinterpret_cast<const uint4*>(ring_g)[i];
        __syncwarp();
    }
    uint8_t* log = region + PKT_LOG_OFF;
    int off = 0;
    const uint32_t nb_cifs = C.geom.nb_cifs;
    bool pushed = false;
    for (uint32_t c = 0; c < nb_cifs; c++) {
        if (!C.msc_valid[(size_t(s) * nb_cifs + c) * C.max_subs + sub]) continue;
        const uint8_t* buf = C.msc_out + (size_t(s) * nb_cifs + c) * CIF_OUT_STRIDE + cfg.out_offset;
        pkt_frame(sh, ring, sh.fec[w], sh.pkt[w], buf, int(cfg.n_out_bytes), use_fec, R, log, off, cap, lane);
        pushed = true;
    }
    if (use_fec && pushed) {
        __syncwarp();
        for (int i = int(lane); i < PKT_RING_BYTES / 16; i += 32) reinterpret_cast<uint4*>(ring_g)[i] = reinterpret_cast<const uint4*>(ring)[i];
    }
    if (lane == 0) { H->rd = R.rd; H->wr = R.wr; H->fill = R.fill; H->last = R.last; H->log_len = off; }
}

__global__ void __launch_bounds__(PKT_WARPS * 32) k_packet(const ChanDev C, uint8_t* __restrict__ pool, const PktItemDev* __restrict__ items, const int n_items) {
    __shared__ PktShared sh;
    dp_load_shared(sh);
    const uint32_t lane = threadIdx.x & 31u;
    for (int wid = int(blockIdx.x * PKT_WARPS + (threadIdx.x >> 5)); wid < n_items; wid += int(gridDim.x * PKT_WARPS)) {
        pkt_work_item(sh, C, pool, items[wid], lane);
        __syncwarp();
    }
}

// Packed output of the packet entries of streams [first, first + n): runs after k_dabplus_pack (which leaves their index entries
// at {0, 0}), one warp per item, the log copied to layout[item] - layout[first stream's row 0].
__global__ void __launch_bounds__(256) k_packet_pack(const uint8_t* __restrict__ pool, const PktItemDev* __restrict__ items, const int n_items,
                                                     const uint64_t* __restrict__ layout, const int first, const int max_subs,
                                                     uint8_t* __restrict__ log, int32_t* __restrict__ index) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t base = layout[size_t(first) * max_subs];
    for (int w = int((blockIdx.x * blockDim.x + threadIdx.x) >> 5); w < n_items; w += int((gridDim.x * blockDim.x) >> 5)) {
        const PktItemDev it = items[w];
        const size_t idx = size_t(it.stream) * max_subs + it.sub, row = (size_t(it.stream) - size_t(first)) * max_subs + it.sub;
        const uint64_t off = layout[idx] - base;
        const uint8_t* region = pool + it.region;
        const int len = reinterpret_cast<const PktHdr*>(region)->log_len;
        dp_copy_bytes(log + off, region + PKT_LOG_OFF, len, lane);
        if (lane == 0) { index[2 * row] = len ? int32_t(off) : 0; index[2 * row + 1] = len; }
    }
}

// Host side.  Regions are never moved while in use except when the pool grows (a table change, after the context synchronised):
// they are addressed by offset.  Released regions are reused by entries of the same size (the size follows from the bytes per
// CIF); the pool neither shrinks nor coalesces them, so a host that retunes packet services over many bitrates keeps at most one
// set of free regions per size it has used, until the context is destroyed.
struct PacketState {
    DevBuf d_pool, d_items;
    size_t pool_used = 0;
    std::map<uint64_t, std::vector<uint64_t>> free_regions;   // region bytes -> offsets
    std::vector<PktItemDev> items;                            // every active packet entry, by stream then index
    uint64_t items_epoch = 0;
};

// A region for a fresh entry (empty ring, no set in progress, empty log).  Call with the context synchronised.
static int pkt_region_acquire(PacketState& P, const uint64_t log_cap, uint64_t* region) {
    const uint64_t bytes = pkt_region_bytes(log_cap);
    std::vector<uint64_t>& fl = P.free_regions[bytes];
    if (!fl.empty()) {
        *region = fl.back();
        fl.pop_back();
    } else {
        if (P.pool_used + bytes > P.d_pool.bytes) {
            DevBuf grown;
            int rc;
            if ((rc = grown.alloc(std::max(size_t(P.pool_used + bytes), 2 * P.d_pool.bytes)))) return rc;
            if (P.pool_used) {
                const cudaError_t e = cudaMemcpy(grown.p, P.d_pool.p, P.pool_used, cudaMemcpyDeviceToDevice);
                if (e != cudaSuccess) {
                    grown.release();
                    return set_error(DABGPU_ERR_CUDA, "packet pool growth: %s", cudaGetErrorString(e));
                }
            }
            P.d_pool.release();
            P.d_pool = grown;
        }
        *region = P.pool_used;
        P.pool_used += bytes;
    }
    const PktHdr h{0, 0, 0, -1, 0, int32_t(log_cap), 0, 0};
    const cudaError_t e = cudaMemcpy(P.d_pool.as<uint8_t>() + *region, &h, sizeof(h), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        P.free_regions[bytes].push_back(*region);
        return set_error(DABGPU_ERR_CUDA, "packet region reset: %s", cudaGetErrorString(e));
    }
    return DABGPU_OK;
}

static void pkt_region_release(PacketState& P, const uint64_t log_cap, const uint64_t region) {
    P.free_regions[pkt_region_bytes(log_cap)].push_back(region);
}

static void packet_destroy(PacketState& P) {
    P.d_pool.release();
    P.d_items.release();
}

// [i0, i1) of the items of streams [first, first + n)
static void pkt_item_range(const PacketState& P, const int first, const int n, size_t* i0, size_t* i1) {
    auto lo = std::lower_bound(P.items.begin(), P.items.end(), uint32_t(first), [](const PktItemDev& a, uint32_t s) { return a.stream < s; });
    auto hi = std::lower_bound(lo, P.items.end(), uint32_t(first + n), [](const PktItemDev& a, uint32_t s) { return a.stream < s; });
    *i0 = size_t(lo - P.items.begin());
    *i1 = size_t(hi - P.items.begin());
}

static int packet_run(PacketState& P, const ChanDev& C, const int first, const int n, const int num_sms, cudaStream_t stream, uint64_t* launches,
                      Profiler& pf) {
    size_t i0, i1;
    pkt_item_range(P, first, n, &i0, &i1);
    if (i1 == i0) return DABGPU_OK;
    const uint32_t items = uint32_t(i1 - i0);
    const uint32_t ctas = std::min((items + PKT_WARPS - 1) / PKT_WARPS, uint32_t(num_sms) * 8u);
    pf.begin(PROF_DABPLUS, stream);
    k_packet<<<ctas, PKT_WARPS * 32, 0, stream>>>(C, P.d_pool.as<uint8_t>(), P.d_items.as<PktItemDev>() + i0, int(items));
    pf.end(stream);
    (*launches)++;
    CUDA_TRY(cudaGetLastError());
    return DABGPU_OK;
}

static int packet_pack(PacketState& P, const uint64_t* d_layout, const int first, const int n, const int max_subs, uint8_t* d_log, int32_t* d_index,
                       cudaStream_t stream, uint64_t* launches, Profiler& pf) {
    size_t i0, i1;
    pkt_item_range(P, first, n, &i0, &i1);
    if (i1 == i0) return DABGPU_OK;
    const uint32_t items = uint32_t(i1 - i0);
    pf.begin(PROF_DABPLUS, stream);
    k_packet_pack<<<(items + 7u) / 8u, 256, 0, stream>>>(P.d_pool.as<uint8_t>(), P.d_items.as<PktItemDev>() + i0, int(items), d_layout, first,
                                                         max_subs, d_log, d_index);
    pf.end(stream);
    (*launches)++;
    CUDA_TRY(cudaGetLastError());
    return DABGPU_OK;
}

// The last decode's log of one packet entry, as stored.
static int packet_get_events(PacketState& P, const uint64_t region, uint8_t* log_host, size_t log_cap, size_t* log_bytes) {
    PktHdr h;
    CUDA_TRY(cudaMemcpy(&h, P.d_pool.as<uint8_t>() + region, sizeof(h), cudaMemcpyDeviceToHost));
    if (size_t(h.log_len) > log_cap) return set_error(DABGPU_ERR_OVERFLOW, "event log buffer too small");
    if (h.log_len > 0) CUDA_TRY(cudaMemcpy(log_host, P.d_pool.as<uint8_t>() + region + PKT_LOG_OFF, size_t(h.log_len), cudaMemcpyDeviceToHost));
    if (log_bytes) *log_bytes = size_t(h.log_len);
    return DABGPU_OK;
}
