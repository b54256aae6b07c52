"""Synthetic DAB/DAB+ ensemble transmitter (numpy) used to feed the receive path.

The reference tree has no encoder that produces decodable ensembles (its
``OFDM_Modulator`` does no channel coding or frequency interleaving, SURVEY.md H6), so this
module restates the transmit side of ETSI EN 300 401 / TS 102 563 with exactly the conventions
the reference *decoder* expects.  Each function cites the decoder code it is the inverse of
(paths relative to /root/reference/vendor/DAB-Radio/src).

It is workload-generation code for tests and ``bench.py``; nothing here runs on the product path.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Optional, Sequence, Tuple

import numpy as np

# --------------------------------------------------------------------------------------------
# Frame geometry (inverse of ofdm/dab_ofdm_params_ref.cpp:10-58 and dab/constants/dab_parameters.h:26-90)
# --------------------------------------------------------------------------------------------


@dataclass(frozen=True)
class ModeParams:
    mode: int
    nb_frame_symbols: int   # incl. PRS, excl. NULL
    nb_symbol_period: int
    nb_null_period: int
    nb_fft: int
    nb_carriers: int
    nb_fic_symbols: int
    nb_cifs: int
    nb_fibs_per_cif: int

    @property
    def nb_cyclic_prefix(self) -> int:
        return self.nb_symbol_period - self.nb_fft

    @property
    def nb_sym_bits(self) -> int:
        return 2 * self.nb_carriers

    @property
    def nb_frame_bits(self) -> int:
        return (self.nb_frame_symbols - 1) * self.nb_sym_bits

    @property
    def nb_fic_bits(self) -> int:
        return self.nb_fic_symbols * self.nb_sym_bits

    @property
    def nb_fib_group_bits(self) -> int:
        return self.nb_fic_bits // self.nb_cifs

    @property
    def nb_frame_samples(self) -> int:
        return self.nb_null_period + self.nb_frame_symbols * self.nb_symbol_period


MODES = {
    1: ModeParams(1, 76, 2552, 2656, 2048, 1536, 3, 4, 3),
    2: ModeParams(2, 76, 638, 664, 512, 384, 3, 1, 3),
    3: ModeParams(3, 153, 319, 345, 256, 192, 8, 1, 4),
    4: ModeParams(4, 76, 1276, 1328, 1024, 768, 3, 2, 3),
}
CIF_BITS = 55296  # 864 capacity units x 64 bits (dab/msc/msc_decoder.cpp:21-23)

# --------------------------------------------------------------------------------------------
# Bit helpers
# --------------------------------------------------------------------------------------------


def bytes_to_bits(b: np.ndarray) -> np.ndarray:
    """MSB-first unpack (decoder packs MSB-first: viterbi_decoder_core.h:223-235)."""
    return np.unpackbits(np.asarray(b, dtype=np.uint8))


def bits_to_bytes(bits: np.ndarray) -> np.ndarray:
    return np.packbits(np.asarray(bits, dtype=np.uint8))


def prbs_bits(n: int) -> np.ndarray:
    """Energy dispersal PRBS x^9+x^5+1, all-ones start (dab/algorithms/additive_scrambler.h:16-28)."""
    reg = 0x1FF
    out = np.empty(n, dtype=np.uint8)
    for i in range(n):
        v = ((reg >> 8) ^ (reg >> 4)) & 1
        out[i] = v
        reg = ((reg << 1) | v) & 0x1FF
    return out


_PRBS_CACHE = prbs_bits(8 * 4096)


def scramble_bits(bits: np.ndarray) -> np.ndarray:
    n = bits.size
    if n > _PRBS_CACHE.size:
        return bits ^ prbs_bits(n)
    return bits ^ _PRBS_CACHE[:n]


def crc16_ccitt(data: np.ndarray, init: int = 0xFFFF, xorout: int = 0xFFFF, poly: int = 0x1021) -> int:
    """MSB-first CRC16 (dab/algorithms/crc.h:26-36; FIB/AU parameters fic_decoder.cpp:19-33)."""
    crc = init
    for byte in np.asarray(data, dtype=np.uint8).tolist():
        crc ^= byte << 8
        for _ in range(8):
            crc = ((crc << 1) ^ poly) & 0xFFFF if (crc & 0x8000) else (crc << 1) & 0xFFFF
    return crc ^ xorout


def firecode(data9: np.ndarray) -> int:
    """Fire code over superframe bytes 2..10 (dab/audio/aac_frame_processor.cpp:74-85, 179-191)."""
    return crc16_ccitt(data9, init=0, xorout=0, poly=0x782F)


# --------------------------------------------------------------------------------------------
# Convolutional code + puncturing (inverse of dab/algorithms/dab_viterbi_decoder.cpp:15-25, 131-181)
# --------------------------------------------------------------------------------------------
# Generator taps as delays (bit k of G = input delayed by k): 109,79,83,109 = octal 133,171,145,133
_G = (109, 79, 83, 109)
_G_TAPS = tuple(tuple(k for k in range(7) if (g >> k) & 1) for g in _G)


def conv_encode(bits: np.ndarray) -> np.ndarray:
    """Rate 1/4 K=7 mother code with 6 zero tail bits; output x0,x1,x2,x3 per input bit."""
    n = bits.size + 6
    hist = np.zeros(n + 6, dtype=np.uint8)
    hist[6:6 + bits.size] = bits
    out = np.zeros((n, 4), dtype=np.uint8)
    for r, taps in enumerate(_G_TAPS):
        acc = np.zeros(n, dtype=np.uint8)
        for k in taps:
            acc ^= hist[6 - k:6 - k + n]
        out[:, r] = acc
    return out.reshape(-1)


_PI_ORDER = (0, 4, 2, 6, 1, 5, 3, 7)


def pi_counts(pi: int) -> Tuple[int, ...]:
    """Kept-bits-per-group form of puncturing vector PI_pi (EN 300 401 table 13; same form as
    dab/constants/puncture_codes.h:42-67).  PI_i keeps 8+i of every 32 mother bits; within a tier
    the extra bits are granted to the 4-bit groups in bit-reversed order."""
    assert 1 <= pi <= 24
    base = 1 + (pi - 1) // 8
    extra = (pi - 1) % 8
    cnt = [base] * 8
    for k in range(extra + 1):
        cnt[_PI_ORDER[k]] += 1
    return tuple(cnt)


PI_X_COUNTS = (2, 2, 2, 2, 2, 2)


def puncture_mask(segments: Sequence[Tuple[int, int]]) -> np.ndarray:
    """segments = [(pi, n_mother_bits)], pi=0 is the 24-bit tail code.  Returns keep mask."""
    masks = []
    for pi, nbits in segments:
        cnt = PI_X_COUNTS if pi == 0 else pi_counts(pi)
        groups = nbits // 4
        c = np.array([cnt[g % len(cnt)] for g in range(groups)], dtype=np.int64)
        m = (np.arange(4)[None, :] < c[:, None]).reshape(-1)
        masks.append(m)
    return np.concatenate(masks)


def eep_segments(length_cu: int, level: int, type_b: bool) -> List[Tuple[int, int]]:
    """EEP schedule (EN 300 401 11.3.2; decoder: dab/msc/msc_decoder.cpp:77-115,
    dab/constants/subchannel_protection_tables.h:121-154).  level is 0-based (0 => 1-A/1-B)."""
    if not type_b:
        if length_cu == 8:  # table quirk the reference applies to ANY type-A sub-channel of 8 CU
            n, lx, pis = 1, (5, 1), (13, 12)
        else:
            mult, eq, pis = [
                (12, ((6, -3), (0, 3)), (24, 23)),
                (8, ((2, -3), (4, 3)), (14, 13)),
                (6, ((6, -3), (0, 3)), (8, 7)),
                (4, ((4, -3), (2, 3)), (3, 2)),
            ][level]
            n = length_cu // mult
            lx = tuple(m * n + b for m, b in eq)
    else:
        mult, pis = [(27, (10, 9)), (21, (6, 5)), (18, (4, 3)), (15, (2, 1))][level]
        n = length_cu // mult
        lx = (24 * n - 3, 3)
    return [(pis[0], 128 * lx[0]), (pis[1], 128 * lx[1]), (0, 24)]


# UEP rows actually exercised by tests: index -> (size CU, L1..L4, PI1..PI4, padding bits)
# (EN 300 401 tables 8/15; decoder: subchannel_protection_tables.h:21-86)
UEP_ROWS = {
    0: (16, (3, 4, 17, 0), (5, 3, 2, 0), 0),
    2: (24, (3, 4, 14, 3), (15, 9, 6, 8), 0),
    4: (35, (3, 5, 13, 3), (24, 17, 12, 17), 4),
    14: (32, (6, 9, 31, 2), (5, 3, 2, 3), 0),
    16: (48, (6, 12, 27, 3), (16, 8, 6, 9), 0),
    37: (140, (11, 20, 62, 3), (24, 17, 13, 19), 8),
    63: (416, (12, 28, 245, 3), (24, 20, 14, 23), 8),
}


def uep_segments(index: int) -> List[Tuple[int, int]]:
    _, ls, pis, _ = UEP_ROWS[index]
    # the reference decoder calls update() for all four segments, PI index 0 never occurs with L>0
    segs = [(pi, 128 * l) for l, pi in zip(ls, pis) if l > 0]
    return segs + [(0, 24)]


def channel_encode(info_bytes: np.ndarray, segments: Sequence[Tuple[int, int]]) -> np.ndarray:
    """energy dispersal -> conv encode -> puncture.  Returns hard bits 0/1."""
    bits = scramble_bits(bytes_to_bits(info_bytes))
    mother = conv_encode(bits)
    mask = puncture_mask(segments)
    assert mask.size == mother.size, (mask.size, mother.size)
    return mother[mask]


FIC_SEGMENTS = [(16, 128 * 21), (15, 128 * 3), (0, 24)]  # dab/fic/fic_decoder.cpp:74-85


def make_fib(payload: bytes) -> np.ndarray:
    """30 data bytes (0xFF padded) + CRC16 (dab/fic/fic_decoder.cpp:98-116)."""
    assert len(payload) <= 30
    data = np.frombuffer(payload + b"\xff" * (30 - len(payload)), dtype=np.uint8)
    crc = crc16_ccitt(data)
    return np.concatenate([data, np.array([crc >> 8, crc & 0xFF], dtype=np.uint8)])


# --------------------------------------------------------------------------------------------
# Sub-channel description
# --------------------------------------------------------------------------------------------


@dataclass
class Subchannel:
    id: int
    start_address: int
    length: int
    is_uep: bool = False
    uep_index: int = 0
    eep_level: int = 2      # 0-based: 2 => 3-A / 3-B
    eep_type_b: bool = False
    dabplus: bool = True    # payload carries DAB+ superframes (needs frame bytes % 24 == 0)

    def segments(self) -> List[Tuple[int, int]]:
        return uep_segments(self.uep_index) if self.is_uep else eep_segments(self.length, self.eep_level, self.eep_type_b)

    @property
    def frame_bytes(self) -> int:
        """decoded bytes per logical frame = steps/8 without the 6 tail bits"""
        return sum(n for _, n in self.segments()[:-1]) // 4 // 8

    @property
    def nb_bits(self) -> int:
        return self.length * 64


def fig0_1(subchannels: Sequence[Subchannel]) -> List[bytes]:
    """FIG 0/1 sub-channel organisation, long form for EEP, short form for UEP
    (parser: dab/fic/fig_processor.cpp:302-365).  Returns FIG blobs (<= 30 bytes each)."""
    figs, body = [], b""
    for sc in subchannels:
        if sc.is_uep:
            e = bytes([(sc.id << 2) | (sc.start_address >> 8), sc.start_address & 0xFF, sc.uep_index & 0x3F])
        else:
            opt = 1 if sc.eep_type_b else 0
            w = (1 << 15) | (opt << 12) | (sc.eep_level << 10) | sc.length
            e = bytes([(sc.id << 2) | (sc.start_address >> 8), sc.start_address & 0xFF, w >> 8, w & 0xFF])
        if len(body) + len(e) > 28:
            figs.append(bytes([(0 << 5) | (len(body) + 1), 0x01]) + body)
            body = b""
        body += e
    if body:
        figs.append(bytes([(0 << 5) | (len(body) + 1), 0x01]) + body)
    return figs


def fig0_2(subchannels: Sequence[Subchannel]) -> List[bytes]:
    """FIG 0/2 service organisation: one programme service (16-bit SId 0xD100 + SubChId) per sub-channel with a single
    primary stream-audio component, ASCTy 63 (DAB+) or 0 (DAB) (parser: dab/fic/fig_processor.cpp:364-487)."""
    figs, body = [], b""
    for sc in subchannels:
        sid = 0xD100 + sc.id
        e = bytes([sid >> 8, sid & 0xFF, 0x01, (0 << 6) | (63 if sc.dabplus else 0), (sc.id << 2) | 0x02])
        if len(body) + len(e) > 28:
            figs.append(bytes([(0 << 5) | (len(body) + 1), 0x02]) + body)
            body = b""
        body += e
    if body:
        figs.append(bytes([(0 << 5) | (len(body) + 1), 0x02]) + body)
    return figs


# --------------------------------------------------------------------------------------------
# RS(120,110) encoder and DAB+ superframe builder
# (inverse of dab/audio/aac_frame_processor.cpp:201-362, reed_solomon_decoder.cpp:70-178)
# --------------------------------------------------------------------------------------------
_GF_EXP = np.zeros(512, dtype=np.int64)
_GF_LOG = np.zeros(256, dtype=np.int64)
_sr = 1
for _i in range(255):
    _GF_EXP[_i] = _sr
    _GF_LOG[_sr] = _i
    _sr <<= 1
    if _sr & 0x100:
        _sr ^= 0x11D
_GF_EXP[255:510] = _GF_EXP[0:255]


def _gf_mul(a: int, b: int) -> int:
    if a == 0 or b == 0:
        return 0
    return int(_GF_EXP[_GF_LOG[a] + _GF_LOG[b]])


def _rs_genpoly(nroots: int = 10) -> List[int]:
    g = [1]
    for i in range(nroots):  # fcr = 0, prim = 1 : roots alpha^0..alpha^(nroots-1)
        root = int(_GF_EXP[i])
        ng = [0] * (len(g) + 1)
        for j, c in enumerate(g):
            ng[j] ^= c               # x * c
            ng[j + 1] ^= _gf_mul(c, root)
        g = ng
    return g  # highest degree first, monic


_RS_G10 = _rs_genpoly(10)
_RS_G16 = _rs_genpoly(16)


def rs_encode(data: Sequence[int], nroots: int = 10) -> List[int]:
    """Systematic shortened RS over GF(2^8)/0x11D: parity = data(x)*x^nroots mod g(x)."""
    g = _RS_G10 if nroots == 10 else _rs_genpoly(nroots)
    rem = [0] * nroots
    for d in data:
        fb = d ^ rem[0]
        rem = rem[1:] + [0]
        if fb:
            for j in range(nroots):
                rem[j] ^= _gf_mul(fb, g[j + 1])
    return rem


def packet_fec_set(rng: np.random.Generator, lengths: Optional[Sequence[int]] = None) -> List[np.ndarray]:
    """One complete packet-mode FEC set (ETSI EN 300 401 5.3.5): data packets filling the 2256-byte application data table,
    then the nine 24-byte FEC packets (address 1022, counters 0..8) that carry the RS(204,188) parity of its 12 rows."""
    if lengths is None:
        lengths, left = [], 2256
        while left > 0:
            n = int(rng.choice([x for x in (24, 48, 72, 96) if x <= left]))
            lengths.append(n)
            left -= n
    assert sum(lengths) == 2256
    packets = []
    for i, n in enumerate(lengths):
        p = rng.integers(0, 256, size=n, dtype=np.uint8)
        address = int(rng.integers(1, 1000))
        p[0] = ((n // 24 - 1) << 6) | ((i & 3) << 4) | (int(rng.integers(0, 4)) << 2) | (address >> 8)
        p[1] = address & 0xFF
        packets.append(p)
    table = np.concatenate(packets)
    parity = np.zeros(192, dtype=np.uint8)
    for y in range(12):
        parity[y::12] = rs_encode([int(v) for v in table[y::12]], 16)
    for i in range(9):
        p = np.zeros(24, dtype=np.uint8)
        p[0] = (i << 2) | 0x03
        p[1] = 0xFE
        n = 22 if i < 8 else 16
        p[2:2 + n] = parity[22 * i:22 * i + n]
        packets.append(p)
    return packets


def build_superframe(bitrate_kbps: int, rng: np.random.Generator, dac_rate: int = 1, sbr: int = 1,
                     stereo: int = 1, ps: int = 0, mpeg: int = 0) -> np.ndarray:
    """One DAB+ audio superframe (5 logical frames) with valid fire code, AU CRCs and RS parity."""
    n_cw = bitrate_kbps // 8
    total = 120 * n_cw
    data_len = 110 * n_cw
    num_aus = {(0, 1): 2, (1, 1): 3, (0, 0): 4, (1, 0): 6}[(dac_rate, sbr)]
    tbl_bits = 12 * (num_aus - 1)
    hdr_len = 3 + (tbl_bits + 7) // 8
    # split the AU area evenly
    au_area = data_len - hdr_len
    base = au_area // num_aus
    starts = [hdr_len + i * base for i in range(num_aus)] + [data_len]
    sf = np.zeros(total, dtype=np.uint8)
    sf[2] = (dac_rate << 6) | (sbr << 5) | (stereo << 4) | (ps << 3) | mpeg
    acc, nacc, pos = 0, 0, 3
    for s in starts[1:num_aus]:
        acc = (acc << 12) | s
        nacc += 12
        while nacc >= 8:
            sf[pos] = (acc >> (nacc - 8)) & 0xFF
            pos += 1
            nacc -= 8
    if nacc:
        sf[pos] = (acc << (8 - nacc)) & 0xFF
    for i in range(num_aus):
        a, b = starts[i], starts[i + 1]
        payload = rng.integers(0, 256, size=b - a - 2, dtype=np.uint8)
        crc = crc16_ccitt(payload)
        sf[a:b - 2] = payload
        sf[b - 2] = crc >> 8
        sf[b - 1] = crc & 0xFF
    fc = firecode(sf[2:11])
    sf[0], sf[1] = fc >> 8, fc & 0xFF
    # RS: codeword i = bytes {i + j*n_cw}
    for i in range(n_cw):
        cw = sf[i:data_len:n_cw].tolist()
        par = rs_encode(cw, 10)
        sf[data_len + i::n_cw] = np.array(par, dtype=np.uint8)
    return sf


# --------------------------------------------------------------------------------------------
# Ensemble multiplexer: FIC + MSC with time interleaving -> hard bits per transmission frame
# --------------------------------------------------------------------------------------------
_TI = np.array([0, 8, 4, 12, 2, 10, 6, 14, 1, 9, 5, 13, 3, 11, 7, 15])  # dab/msc/cif_deinterleaver.cpp:8-11


class EnsembleTx:
    """Generates transmission-frame payload bits for a fixed sub-channel layout.

    ``logical_frames[sc.id]`` accumulates the decoded-domain payload bytes per CIF so tests can
    compare decoder output (which lags 15 CIFs: cif_deinterleaver.cpp:36-71)."""

    def __init__(self, mode: int, subchannels: Sequence[Subchannel], seed: int = 1, fill_random: bool = True):
        self.p = MODES[mode]
        self.subchannels = list(subchannels)
        self.rng = np.random.default_rng(seed)
        self.fill_random = fill_random
        self.cif_count = 0
        self.logical_frames = {sc.id: [] for sc in self.subchannels}
        self.superframes = {sc.id: [] for sc in self.subchannels}
        self.fibs: List[np.ndarray] = []
        self._sf_buf = {sc.id: np.zeros(0, dtype=np.uint8) for sc in self.subchannels}
        # encoded logical frames history for the interleaver: per sub-channel ring of 16
        self._enc_hist = {sc.id: [np.zeros(sc.nb_bits, dtype=np.uint8) for _ in range(16)] for sc in self.subchannels}
        self._figs = fig0_1(self.subchannels) + fig0_2(self.subchannels)
        self._fig_pos = 0

    def _next_logical_frame(self, sc: Subchannel) -> np.ndarray:
        nb = sc.frame_bytes
        if sc.dabplus and nb % 24 == 0:
            buf = self._sf_buf[sc.id]
            if buf.size < nb:
                sf = build_superframe(nb // 3, self.rng)
                self.superframes[sc.id].append(sf)
                buf = np.concatenate([buf, sf])
            frame, self._sf_buf[sc.id] = buf[:nb], buf[nb:]
            return frame
        return self.rng.integers(0, 256, size=nb, dtype=np.uint8)

    def _next_fib_group(self) -> np.ndarray:
        fibs = []
        for _ in range(self.p.nb_fibs_per_cif):
            payload = b""
            if self._figs:
                fig = self._figs[self._fig_pos % len(self._figs)]
                self._fig_pos += 1
                payload = fig
            fibs.append(make_fib(payload))
        self.fibs.extend(fibs)
        return np.concatenate(fibs)

    def next_cif(self) -> np.ndarray:
        cif = self.rng.integers(0, 2, size=CIF_BITS, dtype=np.uint8) if self.fill_random else np.zeros(CIF_BITS, dtype=np.uint8)
        r = self.cif_count
        for sc in self.subchannels:
            info = self._next_logical_frame(sc)
            self.logical_frames[sc.id].append(info)
            enc = channel_encode(info, sc.segments())
            assert enc.size <= sc.nb_bits, (enc.size, sc.nb_bits, sc)
            if enc.size < sc.nb_bits:   # UEP padding bits (EN 300 401 table 15), sent as zeros
                enc = np.concatenate([enc, np.zeros(sc.nb_bits - enc.size, dtype=np.uint8)])
            hist = self._enc_hist[sc.id]
            hist[r % 16] = enc
            # bit i of logical frame r' is sent in CIF r' + T[i%16]  =>  CIF r carries frame r - T[i%16]
            idx = np.arange(sc.nb_bits)
            src = (r - _TI[idx % 16]) % 16
            stacked = np.stack(hist)
            out = stacked[src, idx]
            # frames before the start of time are zeros (hist initialised to zeros)
            a = sc.start_address * 64
            cif[a:a + sc.nb_bits] = out
        self.cif_count += 1
        return cif

    def next_frame_bits(self) -> np.ndarray:
        p = self.p
        if p.mode == 3:
            # FIB group is 4 FIBs = 128 bytes, 3072 punctured bits (not decodable by the reference FIC_Decoder)
            fic = [self.rng.integers(0, 2, size=p.nb_fib_group_bits, dtype=np.uint8) for _ in range(p.nb_cifs)]
        else:
            fic = [channel_encode(self._next_fib_group(), FIC_SEGMENTS) for _ in range(p.nb_cifs)]
        msc = [self.next_cif() for _ in range(p.nb_cifs)]
        bits = np.concatenate(fic + msc)
        assert bits.size == p.nb_frame_bits
        return bits


# --------------------------------------------------------------------------------------------
# OFDM modulator (inverse of ofdm/ofdm_demodulator.cpp:728-739, 842-889)
# --------------------------------------------------------------------------------------------
_PRS_H = np.array([
    [0, 2, 0, 0, 0, 0, 1, 1, 2, 0, 0, 0, 2, 2, 1, 1, 0, 2, 0, 0, 0, 0, 1, 1, 2, 0, 0, 0, 2, 2, 1, 1],
    [0, 3, 2, 3, 0, 1, 3, 0, 2, 1, 2, 3, 2, 3, 3, 0, 0, 3, 2, 3, 0, 1, 3, 0, 2, 1, 2, 3, 2, 3, 3, 0],
    [0, 0, 0, 2, 0, 2, 1, 3, 2, 2, 0, 2, 2, 0, 1, 3, 0, 0, 0, 2, 0, 2, 1, 3, 2, 2, 0, 2, 2, 0, 1, 3],
    [0, 1, 2, 1, 0, 3, 3, 2, 2, 3, 2, 1, 2, 1, 3, 2, 0, 1, 2, 1, 0, 3, 3, 2, 2, 3, 2, 1, 2, 1, 3, 2],
])
# (i, n) per block of 32 carriers, negative carriers first then positive (EN 300 401 table 23 / annex;
# same data as ofdm/dab_prs_ref.cpp:24-131)
_PRS_IN = {
    1: ([(0, 1), (1, 2), (2, 0), (3, 1), (0, 3), (1, 2), (2, 2), (3, 3), (0, 2), (1, 1), (2, 2), (3, 3),
         (0, 1), (1, 2), (2, 3), (3, 3), (0, 2), (1, 2), (2, 2), (3, 1), (0, 1), (1, 3), (2, 1), (3, 2)],
        [(0, 3), (3, 1), (2, 1), (1, 1), (0, 2), (3, 2), (2, 1), (1, 0), (0, 2), (3, 2), (2, 3), (1, 3),
         (0, 0), (3, 2), (2, 1), (1, 3), (0, 3), (3, 3), (2, 3), (1, 0), (0, 3), (3, 0), (2, 1), (1, 1)]),
    2: ([(0, 2), (1, 3), (2, 2), (3, 2), (0, 1), (1, 2)], [(2, 0), (1, 2), (0, 2), (3, 1), (2, 0), (1, 3)]),
    3: ([(0, 2), (1, 3), (2, 0)], [(3, 2), (2, 2), (1, 2)]),
    4: ([(0, 0), (1, 1), (2, 1), (3, 2), (0, 2), (1, 2), (2, 0), (3, 3), (0, 3), (1, 1), (2, 3), (3, 2)],
        [(0, 0), (3, 1), (2, 0), (1, 2), (0, 0), (3, 1), (2, 2), (1, 2), (0, 2), (3, 1), (2, 3), (1, 0)]),
}


def prs_phase_index(mode: int) -> np.ndarray:
    """(h+n) mod 4 for carriers ordered -K/2..-1, +1..+K/2 (phase = pi/2 * value)."""
    neg, pos = _PRS_IN[mode]
    out = []
    for (i, n) in neg:
        out.extend(((_PRS_H[i] + n) % 4).tolist())
    for (i, n) in pos:
        out.extend(((_PRS_H[i] + n) % 4).tolist())
    return np.array(out, dtype=np.int64)


def carrier_map(nb_fft: int, nb_carriers: int) -> np.ndarray:
    """Frequency interleaver (EN 300 401 14.6.1; decoder table ofdm/dab_mapper_ref.cpp:10-50)."""
    pi = np.zeros(nb_fft, dtype=np.int64)
    for i in range(1, nb_fft):
        pi[i] = (13 * pi[i - 1] + nb_fft // 4 - 1) % nb_fft
    dc = nb_fft // 2
    lo, hi = dc - nb_carriers // 2, dc + nb_carriers // 2
    out = []
    for v in pi.tolist():
        if v < lo or v > hi or v == dc:
            continue
        out.append(v - lo if v < dc else v - lo - 1)
    return np.array(out, dtype=np.int64)


def ofdm_modulate(frames_bits: Sequence[np.ndarray], mode: int) -> np.ndarray:
    """Returns complex64 baseband: [NULL | PRS | data symbols] per frame, unit-power carriers."""
    p = MODES[mode]
    K, N = p.nb_carriers, p.nb_fft
    cmap = carrier_map(N, K)
    # fft bin of carrier slot s (slots ordered -K/2..-1, +1..+K/2)
    slot_k = np.concatenate([np.arange(-K // 2, 0), np.arange(1, K // 2 + 1)])
    slot_bin = slot_k % N
    prs = np.exp(1j * np.pi / 2 * prs_phase_index(mode))
    out = []
    for bits in frames_bits:
        sym_bits = bits.reshape(p.nb_frame_symbols - 1, 2 * K)
        cur = prs.copy()
        spectra = np.zeros((p.nb_frame_symbols, N), dtype=np.complex128)
        spectra[0, slot_bin] = cur
        for l in range(p.nb_frame_symbols - 1):
            b0 = sym_bits[l, :K].astype(np.float64)
            b1 = sym_bits[l, K:].astype(np.float64)
            q_pair = ((1 - 2 * b0) + 1j * (1 - 2 * b1)) / np.sqrt(2.0)
            q = np.empty(K, dtype=np.complex128)
            q[cmap] = q_pair          # pair n sits on carrier slot cmap[n]
            cur = cur * q
            spectra[l + 1, slot_bin] = cur
        t = np.fft.ifft(spectra, axis=1) * (N / np.sqrt(K))   # unit average power
        syms = np.concatenate([t[:, N - p.nb_cyclic_prefix:], t], axis=1).reshape(-1)
        out.append(np.zeros(p.nb_null_period, dtype=np.complex128))
        out.append(syms)
    return np.concatenate(out).astype(np.complex64)


def impair(iq: np.ndarray, snr_db: Optional[float], cfo_norm: float, lead_samples: int, seed: int,
           tail_samples: int = 0) -> np.ndarray:
    """AWGN (signal power 1 during symbols), CFO (cycles/sample), leading/trailing noise-only samples."""
    rng = np.random.default_rng(seed)
    x = np.concatenate([np.zeros(lead_samples, np.complex64), iq, np.zeros(tail_samples, np.complex64)])
    n = np.arange(x.size, dtype=np.float64)
    x = x * np.exp(2j * np.pi * cfo_norm * n)
    if snr_db is not None:
        sigma = np.sqrt(0.5 * 10 ** (-snr_db / 10))
        x = x + sigma * (rng.standard_normal(x.size) + 1j * rng.standard_normal(x.size))
    return x.astype(np.complex64)


def to_u8(iq: np.ndarray, rms_lsb: float = 30.0) -> np.ndarray:
    """u8 = clamp(trunc(x*s + 127.5)) I,Q interleaved (examples/app_helpers/app_iq_readers.h:51-63)."""
    v = np.empty(iq.size * 2, dtype=np.float32)
    v[0::2] = iq.real
    v[1::2] = iq.imag
    v = v * np.float32(rms_lsb) + np.float32(127.5)   # unit-power signal => |x| RMS = rms_lsb LSB
    return np.clip(np.trunc(v), 0, 255).astype(np.uint8)


def hard_to_soft(bits: np.ndarray, rng: Optional[np.random.Generator] = None, snr_db: Optional[float] = None,
                 amplitude: float = 127.0) -> np.ndarray:
    """0/1 -> int8 soft decisions (+127 = logical 1, viterbi_config.h:11-14) with optional AWGN."""
    x = (2.0 * bits.astype(np.float64) - 1.0)
    if snr_db is not None:
        assert rng is not None
        x = x + rng.standard_normal(x.size) * np.sqrt(0.5 * 10 ** (-snr_db / 10))
        x = np.clip(x * (amplitude / 2.0), -127, 127)   # nominal level at half scale so noise is not all clipped
    else:
        x = x * amplitude
    return np.trunc(x).astype(np.int8)


def default_ensemble() -> List[Subchannel]:
    """Config 1 of SURVEY.md 8(d): 18 DAB+ sub-channels EEP 3-A 48 CU filling 864 CU."""
    return [Subchannel(id=i, start_address=48 * i, length=48, eep_level=2, eep_type_b=False) for i in range(18)]


def periodic_frames(mode: int, subchannels: Sequence[Subchannel], seed: int, period_frames: int, return_logical: bool = False):
    """[period_frames, nb_frame_bits] coded transmission frames whose endless repetition is a valid transmission: the logical
    frames of every sub-channel repeat with the period (a whole number of 5-CIF DAB+ superframes), hence so do the
    time-interleaved CIFs once the 16-CIF interleaver has filled.  Used to feed throughput runs of any length from a short buffer.
    return_logical: also return {sub-channel id: [period_cifs, frame_bytes]} = the bytes a decoder must give back, one period of them."""
    p = MODES[mode]
    period_cifs = period_frames * p.nb_cifs
    assert period_cifs % 5 == 0 and period_cifs >= 16, "the period must hold whole superframes and at least the interleaver depth"
    ens = EnsembleTx(mode, subchannels, seed=seed, fill_random=False)
    cache = {sc.id: [] for sc in ens.subchannels}
    fresh = ens._next_logical_frame

    def replay(sc: Subchannel) -> np.ndarray:
        if ens.cif_count < period_cifs:
            cache[sc.id].append(fresh(sc))
            return cache[sc.id][-1]
        return cache[sc.id][ens.cif_count % period_cifs]

    ens._next_logical_frame = replay
    frames = [ens.next_frame_bits() for _ in range(2 * period_frames)]
    if return_logical:
        return np.stack(frames[period_frames:]), {k: np.stack(v) for k, v in cache.items()}
    return np.stack(frames[period_frames:])


def wideband_capture(mode: int, ensembles: Sequence[np.ndarray], D: int, offsets_hz: Sequence[int], snr_db: float = 15.0,
                     cfo_hz: Sequence[float] = (), shifts: Sequence[int] = (), gains_db: Sequence[float] = (), seed: int = 0,
                     mask_hz: float = 800e3, sample_rate: Optional[int] = None) -> np.ndarray:
    """One period of a periodic multi-ensemble capture at D x 2.048 MS/s, or at sample_rate Hz when given (then D is ignored; the
    period must be a whole number of samples at that rate, as it is for 5 Mode I frames at every multiple of 25 Hz)
    (complex128; np.take(..., mode="wrap") continues it).
    ensembles[k] = the coded frames of one period of periodic_frames(); ensemble k gets AWGN at snr_db, a band limit of
    +-mask_hz (a transmitter's spectrum mask), a CFO of cfo_hz[k] and a time shift of shifts[k] samples (both cyclic), the gain
    gains_db[k], and sits offsets_hz[k] above the capture centre.  Built in the frequency domain over the whole period, so the
    CFO and the offsets are rounded to the period's bin spacing (2.048 MHz / period samples, about 2 Hz)."""
    p = MODES[mode]
    L = len(ensembles[0]) * p.nb_frame_samples
    if sample_rate is None:
        M, scale = D * L, D
    else:
        assert (L * sample_rate) % 2048000 == 0, "the period is not a whole number of samples at this rate"
        M = L * sample_rate // 2048000
        scale = M / L
    Y = np.zeros(M, dtype=np.complex128)
    fb = np.fft.fftfreq(L, 1.0 / L).astype(np.int64)
    keep = np.nonzero(np.abs(fb) * 2048000.0 / L <= mask_hz)[0]
    rng = np.random.default_rng(seed)
    sigma = np.sqrt(0.5 * 10 ** (-snr_db / 10))
    for k, f in enumerate(offsets_hz):
        x = ofdm_modulate(list(ensembles[k]), mode).astype(np.complex128)
        assert x.size == L
        x = x + sigma * (rng.standard_normal(L) + 1j * rng.standard_normal(L))
        if k < len(shifts):
            x = np.roll(x, shifts[k])
        X = np.fft.fft(x)
        shift = int(round(f * L / 2048000.0)) + (int(round(cfo_hz[k] * L / 2048000.0)) if k < len(cfo_hz) else 0)
        g = 10 ** ((gains_db[k] if k < len(gains_db) else 0.0) / 20)
        np.add.at(Y, (fb[keep] + shift) % M, X[keep] * (scale * g))
    return np.fft.ifft(Y)


def quantize(iq: np.ndarray, fmt: str, rms: float) -> np.ndarray:
    """complex samples scaled to `rms` (LSB, or full scale for raw_f32l) -> raw interleaved I,Q of a reader mode
    (examples/app_helpers/app_iq_readers.h); values beyond the format's range clip."""
    v = np.empty(iq.size * 2, dtype=np.float64)
    v[0::2], v[1::2] = iq.real, iq.imag
    v *= rms / np.sqrt(np.mean(np.abs(iq) ** 2))
    if fmt == "raw_u8":
        return np.clip(np.round(v + 127.5), 0, 255).astype(np.uint8)
    if fmt == "raw_s8":
        return np.clip(np.round(v), -127, 127).astype(np.int8)
    if fmt == "raw_s16l":
        return np.clip(np.round(v), -32767, 32767).astype("<i2")
    return v.astype("<f4")
