"""ctypes bindings for the two CPU oracles.  TEST INFRASTRUCTURE, not product code.

  * ``RefLib``  -> oracle/_ref/libdabref.so   : the unmodified reference classes (oracle/ref_harness.cpp)
  * ``PortLib`` -> oracle/_ref/libdaboracle.so: the plain-C restatement (oracle/dab_oracle.c)

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this.
"""
from __future__ import annotations

import ctypes as C
import os
import struct
from typing import List, Optional, Sequence, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
REF_SO = os.path.join(_HERE, "_ref", "libdabref.so")
PORT_SO = os.path.join(_HERE, "_ref", "libdaboracle.so")

_i8p = np.ctypeslib.ndpointer(dtype=np.int8, flags="C_CONTIGUOUS")
_u8p = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")


def ref_available() -> bool:
    return os.path.exists(REF_SO)


def port_available() -> bool:
    return os.path.exists(PORT_SO)


class RefLib:
    """The reference's own code (compiled in place from /root/reference by oracle/Makefile)."""

    _inst = None

    @classmethod
    def get(cls) -> "RefLib":
        if cls._inst is None:
            cls._inst = cls()
        return cls._inst

    def __init__(self):
        L = C.CDLL(REF_SO)
        self.L = L
        L.ref_build_info.restype = C.c_char_p
        L.ref_vit_create.restype = C.c_void_p
        L.ref_vit_destroy.argtypes = [C.c_void_p]
        L.ref_vit_decode.argtypes = [C.c_void_p, _i8p, C.c_int, _i32p, _i32p, C.c_int, _u8p, C.c_int, C.POINTER(C.c_uint64)]
        L.ref_vit_decode.restype = C.c_int
        L.ref_scrambler_bytes.argtypes = [_u8p, C.c_int]
        L.ref_fic_create.argtypes = [C.c_int, C.c_int]
        L.ref_fic_create.restype = C.c_void_p
        L.ref_fic_destroy.argtypes = [C.c_void_p]
        L.ref_fic_decode_group.argtypes = [C.c_void_p, _i8p, C.c_int, C.c_int, _u8p, C.c_int]
        L.ref_fic_decode_group.restype = C.c_int
        L.ref_msc_create.argtypes = [C.c_int] * 6
        L.ref_msc_create.restype = C.c_void_p
        L.ref_msc_destroy.argtypes = [C.c_void_p]
        L.ref_msc_decode_cif.argtypes = [C.c_void_p, _i8p, C.c_int, _u8p, C.c_int]
        L.ref_msc_decode_cif.restype = C.c_int
        L.ref_deint_create.argtypes = [C.c_int]
        L.ref_deint_create.restype = C.c_void_p
        L.ref_deint_destroy.argtypes = [C.c_void_p]
        L.ref_deint_push.argtypes = [C.c_void_p, _i8p, _i8p]
        L.ref_deint_push.restype = C.c_int
        L.ref_rs_create.argtypes = [C.c_int] * 6
        L.ref_rs_create.restype = C.c_void_p
        L.ref_rs_destroy.argtypes = [C.c_void_p]
        L.ref_rs_decode.argtypes = [C.c_void_p, _u8p, _i32p, C.c_int]
        L.ref_rs_decode.restype = C.c_int
        L.ref_aac_create.restype = C.c_void_p
        L.ref_aac_destroy.argtypes = [C.c_void_p]
        L.ref_aac_process.argtypes = [C.c_void_p, _u8p, C.c_int, _u8p, C.c_int]
        L.ref_aac_process.restype = C.c_int
        L.ref_ofdm_params.argtypes = [C.c_int, _i32p]
        L.ref_prs_fft.argtypes = [C.c_int, _f32p, C.c_int]
        L.ref_carrier_map.argtypes = [C.c_int, C.c_int, _i32p]
        L.ref_dab_params.argtypes = [C.c_int, _i32p]
        L.ref_ofdm_create.argtypes = [C.c_int, C.c_int]
        L.ref_ofdm_create.restype = C.c_void_p
        L.ref_ofdm_destroy.argtypes = [C.c_void_p]
        L.ref_ofdm_keep_frames.argtypes = [C.c_void_p, C.c_int]
        L.ref_ofdm_frame_bits.argtypes = [C.c_void_p]
        L.ref_ofdm_process_c32.argtypes = [C.c_void_p, _f32p, C.c_int, C.c_int]
        L.ref_ofdm_process_u8.argtypes = [C.c_void_p, _u8p, C.c_int, C.c_int]
        L.ref_ofdm_flush.argtypes = [C.c_void_p]
        L.ref_ofdm_frames_available.argtypes = [C.c_void_p]
        L.ref_ofdm_pop_frame.argtypes = [C.c_void_p, _i8p, _f32p, _i32p]
        L.ref_ofdm_get_state.argtypes = [C.c_void_p, _i32p, _f32p]
        L.ref_ofdm_reset.argtypes = [C.c_void_p]
        L.ref_ofdm_set_coarse_enabled.argtypes = [C.c_void_p, C.c_int]
        if hasattr(L, "ref_ofdm_set_config"):
            L.ref_ofdm_set_config.argtypes = [C.c_void_p, _f32p, _i32p]
        L.ref_ofdm_get_frame_fft.argtypes = [C.c_void_p, _f32p, C.c_int]
        L.ref_ofdm_get_impulse_response.argtypes = [C.c_void_p, _f32p, C.c_int]
        if hasattr(L, "ref_ofdm_get_correlation_buffer"):
            L.ref_ofdm_get_correlation_buffer.argtypes = [C.c_void_p, _f32p, C.c_int]
        if hasattr(L, "ref_ofdm_get_frame_data_vec"):
            L.ref_ofdm_get_frame_data_vec.argtypes = [C.c_void_p, _f32p, C.c_int]
        L.ref_ofdm_get_coarse_response.argtypes = [C.c_void_p, _f32p, C.c_int]
        L.ref_time_ofdm_u8.argtypes = [C.c_int, _u8p, C.c_long, C.c_int, C.c_int, C.POINTER(C.c_int)]
        L.ref_time_ofdm_u8.restype = C.c_double
        if hasattr(L, "ref_time_chain_u8"):
            L.ref_time_chain_u8.argtypes = [C.c_int, _u8p, C.c_long, C.c_int, C.c_int, np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS"), C.c_int,
                                            np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")]
            L.ref_time_chain_u8.restype = C.c_double
        if hasattr(L, "ref_time_chain_split_u8"):
            L.ref_time_chain_split_u8.argtypes = [C.c_int, _u8p, C.c_long, C.c_int, C.c_int, np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS"), C.c_int,
                                                  np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS"),
                                                  np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")]
            L.ref_time_chain_split_u8.restype = C.c_double

        if hasattr(L, "ref_iq_convert"):
            L.ref_iq_convert.argtypes = [C.c_char_p, _u8p, C.c_size_t, _f32p, C.c_size_t]
            L.ref_iq_convert.restype = C.c_long
            L.ref_softbits_to_bytes.argtypes = [_i8p, C.c_size_t, _u8p]
            L.ref_bytes_to_softbits.argtypes = [_u8p, C.c_size_t, _i8p]
        if hasattr(L, "ref_pktfec_create"):
            L.ref_pktfec_create.restype = C.c_void_p
            L.ref_pktfec_destroy.argtypes = [C.c_void_p]
            L.ref_pktfec_read_packet.argtypes = [C.c_void_p, _u8p, C.c_int, _u8p, C.c_int, C.POINTER(C.c_int)]
            L.ref_pktfec_read_packet.restype = C.c_long
        if hasattr(L, "ref_fig_create"):
            L.ref_fig_create.restype = C.c_void_p
            L.ref_fig_destroy.argtypes = [C.c_void_p]
            L.ref_fig_process_fib.argtypes = [C.c_void_p, _u8p]
            L.ref_fig_dump.argtypes = [C.c_void_p, _i32p, C.c_int, _i32p, C.c_int, C.POINTER(C.c_int)]
            L.ref_fig_dump.restype = C.c_int

    def build_info(self) -> str:
        return self.L.ref_build_info().decode()


def _segs(segments: Sequence[Tuple[int, int]]):
    pi = np.ascontiguousarray([s[0] for s in segments], dtype=np.int32)
    nb = np.ascontiguousarray([s[1] for s in segments], dtype=np.int32)
    return pi, nb


class RefViterbi:
    def __init__(self):
        self.lib = RefLib.get().L
        self.h = self.lib.ref_vit_create()

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.ref_vit_destroy(self.h)
            self.h = None

    def decode(self, soft: np.ndarray, segments: Sequence[Tuple[int, int]]) -> Tuple[np.ndarray, int, int]:
        """returns (bytes, consumed, path_error)"""
        soft = np.ascontiguousarray(soft, dtype=np.int8)
        pi, nb = _segs(segments)
        steps = int(nb.sum()) // 4
        n_out = (steps - 6) // 8
        out = np.zeros(n_out, dtype=np.uint8)
        err = C.c_uint64(0)
        consumed = self.lib.ref_vit_decode(self.h, soft, soft.size, pi, nb, len(segments), out, n_out, C.byref(err))
        if consumed < 0:
            raise ValueError("ref_vit_decode: bad arguments")
        return out, consumed, err.value


def ref_scrambler_bytes(n: int) -> np.ndarray:
    out = np.zeros(n, dtype=np.uint8)
    RefLib.get().L.ref_scrambler_bytes(out, n)
    return out


class RefFic:
    def __init__(self, nb_encoded_bits: int = 2304, nb_fibs_per_group: int = 3):
        self.lib = RefLib.get().L
        self.h = self.lib.ref_fic_create(nb_encoded_bits, nb_fibs_per_group)
        self.nb_bits = nb_encoded_bits

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.ref_fic_destroy(self.h)
            self.h = None

    def decode_group(self, bits: np.ndarray, cif_index: int = 0) -> List[bytes]:
        bits = np.ascontiguousarray(bits, dtype=np.int8)
        out = np.zeros(30 * 8, dtype=np.uint8)
        n = self.lib.ref_fic_decode_group(self.h, bits, bits.size, cif_index, out, 8)
        return [out[i * 30:(i + 1) * 30].tobytes() for i in range(n)]


class RefMsc:
    def __init__(self, start_address: int, length: int, is_uep: bool = False, uep_index: int = 0,
                 eep_level: int = 2, eep_type_b: bool = False):
        self.lib = RefLib.get().L
        self.h = self.lib.ref_msc_create(start_address, length, int(is_uep), uep_index, eep_level, int(eep_type_b))
        self.cap = length * 8

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.ref_msc_destroy(self.h)
            self.h = None

    def decode_cif(self, cif_bits: np.ndarray) -> np.ndarray:
        cif_bits = np.ascontiguousarray(cif_bits, dtype=np.int8)
        out = np.zeros(self.cap, dtype=np.uint8)
        n = self.lib.ref_msc_decode_cif(self.h, cif_bits, cif_bits.size, out, self.cap)
        if n < 0:
            raise ValueError("output capacity too small")
        return out[:n].copy()


class RefDeinterleaver:
    def __init__(self, nb_bytes: int):
        self.lib = RefLib.get().L
        self.h = self.lib.ref_deint_create(nb_bytes)
        self.nb_bits = nb_bytes * 8

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.ref_deint_destroy(self.h)
            self.h = None

    def push(self, bits: np.ndarray) -> Optional[np.ndarray]:
        bits = np.ascontiguousarray(bits, dtype=np.int8)
        out = np.zeros(self.nb_bits, dtype=np.int8)
        ok = self.lib.ref_deint_push(self.h, bits, out)
        return out if ok else None


class RefRS:
    def __init__(self, nroots: int = 10, pad: int = 135, gfpoly: int = 0x11D, fcr: int = 0, prim: int = 1):
        self.lib = RefLib.get().L
        self.h = self.lib.ref_rs_create(8, gfpoly, fcr, prim, nroots, pad)
        self.n = 255 - pad
        self.nroots = nroots

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.ref_rs_destroy(self.h)
            self.h = None

    def decode(self, data: np.ndarray) -> Tuple[int, np.ndarray, np.ndarray]:
        """returns (count, corrected data, error positions incl. pad)"""
        d = np.ascontiguousarray(data, dtype=np.uint8).copy()
        pos = np.zeros(self.nroots, dtype=np.int32)
        cnt = self.lib.ref_rs_decode(self.h, d, pos, 0)
        return cnt, d, pos[:max(cnt, 0)].copy()


EV_FIRECODE_ERROR, EV_RS_ERROR, EV_HEADER, EV_AU_CRC_ERROR, EV_AU = 1, 2, 3, 4, 5


def parse_event_log(buf: bytes) -> List[tuple]:
    out, off = [], 0
    while off < len(buf):
        t, a, b, c, d, n = struct.unpack_from("<6i", buf, off)
        off += 24
        payload = bytes(buf[off:off + n])
        off += (n + 3) & ~3
        out.append((t, a, b, c, d, payload))
    return out


class RefAac:
    def __init__(self):
        self.lib = RefLib.get().L
        self.h = self.lib.ref_aac_create()
        self.log = np.zeros(1 << 16, dtype=np.uint8)

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.ref_aac_destroy(self.h)
            self.h = None

    def process(self, frame: np.ndarray) -> List[tuple]:
        frame = np.ascontiguousarray(frame, dtype=np.uint8)
        n = self.lib.ref_aac_process(self.h, frame, frame.size, self.log, self.log.size)
        assert n <= self.log.size
        return parse_event_log(self.log[:n].tobytes())


def parse_packet_log(buf: bytes) -> List[Tuple[bytes, bool]]:
    """flat callback log of the packet-mode FEC processors -> [(packet bytes, is_corrected)]"""
    out, off = [], 0
    while off + 8 <= len(buf):
        n, corrected = np.frombuffer(buf, dtype="<i4", count=2, offset=off)
        off += 8
        out.append((bytes(buf[off:off + int(n)]), bool(corrected)))
        off += (int(n) + 3) & ~3
    return out


class RefPacketFec:
    """MSC_Reed_Solomon_Data_Packet_Processor of the reference build (msc_reed_solomon_data_packet_processor.cpp)."""

    def __init__(self):
        self.lib = RefLib.get().L
        self.h = self.lib.ref_pktfec_create()

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.ref_pktfec_destroy(self.h)
            self.h = None

    def read_packet(self, buf: np.ndarray) -> Tuple[int, List[Tuple[bytes, bool]]]:
        b = np.ascontiguousarray(buf, dtype=np.uint8)
        if b.size == 0:
            b = np.zeros(1, dtype=np.uint8)[:0].copy()
        log = np.zeros(1 << 16, dtype=np.uint8)
        n = C.c_int(0)
        used = self.lib.ref_pktfec_read_packet(self.h, b if b.size else np.zeros(1, dtype=np.uint8), int(buf.size), log, log.size, C.byref(n))
        assert used >= 0
        return int(used), parse_packet_log(log[:n.value].tobytes())


def ref_iq_convert(mode: str, raw: np.ndarray) -> np.ndarray:
    """The reference's reader chain (app_iq_readers.h) over a memory buffer -> complex64."""
    raw = np.ascontiguousarray(raw, dtype=np.uint8)
    out = np.zeros(raw.size + 8, dtype=np.float32)
    n = RefLib.get().L.ref_iq_convert(mode.encode(), raw, raw.size, out, out.size)
    if n < 0:
        raise ValueError(f"reference rejected mode {mode}")
    return out[:n].view(np.complex64).copy()


def ref_softbits_to_bytes(bits: np.ndarray) -> np.ndarray:
    bits = np.ascontiguousarray(bits, dtype=np.int8)
    out = np.zeros(bits.size // 8, dtype=np.uint8)
    RefLib.get().L.ref_softbits_to_bytes(bits, out.size, out)
    return out


def ref_bytes_to_softbits(b: np.ndarray) -> np.ndarray:
    b = np.ascontiguousarray(b, dtype=np.uint8)
    out = np.zeros(b.size * 8, dtype=np.int8)
    RefLib.get().L.ref_bytes_to_softbits(b, b.size, out)
    return out


class RefFig:
    """FIG_Processor -> Radio_FIG_Handler -> DAB_Database_Updater of the reference; dump() returns (subchannels, components)
    in the row formats of dabgpu_autocfg_dump."""

    def __init__(self):
        self.L = RefLib.get().L
        self.h = self.L.ref_fig_create()

    def __del__(self):
        if getattr(self, "h", None):
            self.L.ref_fig_destroy(self.h)
            self.h = None

    def process_fib(self, fib: np.ndarray):
        fib = np.ascontiguousarray(fib[:30], dtype=np.uint8)
        assert fib.size == 30
        self.L.ref_fig_process_fib(self.h, fib)

    def dump(self):
        subs = np.zeros((64, 9), dtype=np.int32)
        comps = np.zeros((256, 10), dtype=np.int32)
        nc = C.c_int(0)
        ns = self.L.ref_fig_dump(self.h, subs.reshape(-1), 64, comps.reshape(-1), 256, C.byref(nc))
        return subs[:ns].copy(), comps[:nc.value].copy()


class RefOfdm:
    STATES = ["FINDING_NULL_POWER_DIP", "READING_NULL_AND_PRS", "RUNNING_COARSE_FREQ_SYNC", "RUNNING_FINE_TIME_SYNC", "READING_SYMBOLS"]

    def __init__(self, mode: int = 1, nb_threads: int = 1):
        self.lib = RefLib.get().L
        self.h = self.lib.ref_ofdm_create(mode, nb_threads)
        if not self.h:
            raise ValueError(f"invalid transmission mode {mode}")
        self.frame_bits = self.lib.ref_ofdm_frame_bits(self.h)
        self.config = dict(OFDM_DEFAULTS)

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.ref_ofdm_destroy(self.h)
            self.h = None

    def set_config(self, **kw):
        """OFDM_Demod::GetConfig() edited between Process() calls; keywords as DabGpu.ofdm_set_config, unnamed knobs keep
        their current values."""
        self.config = _merge_config(self.config, kw)
        c = self.config
        f8 = np.array([c[k] for k in ("signal_l1_update_beta", "null_thresh_start", "null_thresh_end", "fine_freq_update_beta",
                                      "max_coarse_freq_correction_norm", "coarse_freq_slow_beta", "impulse_peak_threshold_db",
                                      "impulse_peak_distance_probability")], dtype=np.float32)
        i3 = np.array([c["signal_l1_nb_samples"], c["signal_l1_nb_decimate"], c["is_coarse_freq_correction"]], dtype=np.int32)
        self.lib.ref_ofdm_set_config(self.h, f8, i3)

    def process_u8(self, iq_u8: np.ndarray, serial: bool = True):
        iq_u8 = np.ascontiguousarray(iq_u8, dtype=np.uint8)
        self.lib.ref_ofdm_process_u8(self.h, iq_u8, iq_u8.size // 2, int(serial))

    def process_c32(self, iq: np.ndarray, serial: bool = True):
        f = np.ascontiguousarray(iq, dtype=np.complex64).view(np.float32)
        self.lib.ref_ofdm_process_c32(self.h, f, f.size // 2, int(serial))

    def flush(self):
        self.lib.ref_ofdm_flush(self.h)

    def pop_frames(self) -> List[Tuple[np.ndarray, float, float, int]]:
        out = []
        while True:
            bits = np.zeros(self.frame_bits, dtype=np.int8)
            cf = np.zeros(2, dtype=np.float32)
            to = np.zeros(1, dtype=np.int32)
            if not self.lib.ref_ofdm_pop_frame(self.h, bits, cf, to):
                break
            out.append((bits, float(cf[0]), float(cf[1]), int(to[0])))
        return out

    def state(self) -> dict:
        s = np.zeros(4, dtype=np.int32)
        f = np.zeros(3, dtype=np.float32)
        self.lib.ref_ofdm_get_state(self.h, s, f)
        return dict(state=int(s[0]), frames_read=int(s[1]), frames_desync=int(s[2]), fine_time_offset=int(s[3]),
                    signal_avg=float(f[0]), coarse=float(f[1]), fine=float(f[2]))

    def frame_fft(self, n_complex: int) -> np.ndarray:
        out = np.zeros(2 * n_complex, dtype=np.float32)
        self.lib.ref_ofdm_get_frame_fft(self.h, out, n_complex)
        return out.view(np.complex64)

    def frame_data_vec(self, n_complex: int) -> np.ndarray:
        out = np.zeros(2 * n_complex, dtype=np.float32)
        self.lib.ref_ofdm_get_frame_data_vec(self.h, out, n_complex)
        return out.view(np.complex64)

    def correlation_buffer(self, n_complex: int) -> np.ndarray:
        out = np.zeros(2 * n_complex, dtype=np.float32)
        n = self.lib.ref_ofdm_get_correlation_buffer(self.h, out, n_complex)
        return out.view(np.complex64)[:n]

    def impulse_response(self, n: int) -> np.ndarray:
        out = np.zeros(n, dtype=np.float32)
        self.lib.ref_ofdm_get_impulse_response(self.h, out, n)
        return out

    def coarse_response(self, n: int) -> np.ndarray:
        out = np.zeros(n, dtype=np.float32)
        self.lib.ref_ofdm_get_coarse_response(self.h, out, n)
        return out


class OfdmConfig(C.Structure):
    """dabo_ofdm_config = dabgpu_ofdm_config (include/dabgpu.h): OFDM_Demod_Config, ofdm_demodulator.h:24-45"""
    _fields_ = [("signal_l1_update_beta", C.c_float), ("signal_l1_nb_samples", C.c_int), ("signal_l1_nb_decimate", C.c_int),
                ("null_thresh_start", C.c_float), ("null_thresh_end", C.c_float), ("fine_freq_update_beta", C.c_float),
                ("is_coarse_freq_correction", C.c_int), ("max_coarse_freq_correction_norm", C.c_float),
                ("coarse_freq_slow_beta", C.c_float), ("impulse_peak_threshold_db", C.c_float),
                ("impulse_peak_distance_probability", C.c_float)]


OFDM_DEFAULTS = dict(signal_l1_update_beta=0.95, signal_l1_nb_samples=100, signal_l1_nb_decimate=5, null_thresh_start=0.35,
                     null_thresh_end=0.75, fine_freq_update_beta=0.9, is_coarse_freq_correction=1,
                     max_coarse_freq_correction_norm=0.5, coarse_freq_slow_beta=0.1, impulse_peak_threshold_db=20.0,
                     impulse_peak_distance_probability=0.15)


def _merge_config(cur: dict, kw: dict) -> dict:
    unknown = set(kw) - set(OFDM_DEFAULTS)
    if unknown:
        raise KeyError(f"unknown OFDM knobs {sorted(unknown)}")
    return {**cur, **kw}


def ofdm_process_call(o, iq: np.ndarray, block_size: int, u8: bool = True) -> None:
    """Feeds the OFDM oracle `o` one call as dabgpu_ofdm_process(n_samples, block_size) presents it: consecutive Process()
    blocks of block_size samples (<= 0: one block), the last one partial; the next call starts a new block."""
    n = iq.size // 2 if u8 else iq.size
    bs = block_size if block_size > 0 else n
    for off in range(0, n, bs):
        end = min(n, off + bs)
        if u8:
            o.process_u8(iq[2 * off:2 * end])
        else:
            o.process_c32(iq[off:end])


def ref_tables(mode: int):
    L = RefLib.get().L
    p = np.zeros(6, dtype=np.int32)
    if L.ref_ofdm_params(mode, p) != 0:
        raise ValueError("invalid mode")
    nb_fft, nb_car = int(p[4]), int(p[5])
    prs = np.zeros(2 * nb_fft, dtype=np.float32)
    L.ref_prs_fft(mode, prs, nb_fft)
    cmap = np.zeros(nb_car, dtype=np.int32)
    L.ref_carrier_map(nb_fft, nb_car, cmap)
    dp = np.zeros(13, dtype=np.int32)
    L.ref_dab_params(mode, dp)
    return p, prs.view(np.complex64), cmap, dp


# =============================================================================================
# Plain-C restatement (oracle/dab_oracle.c)
# =============================================================================================
def _refresh_port() -> None:
    """Brings oracle/_ref/libdaboracle.so up to date with dab_oracle.c before the first load: make rebuilds it when the sources
    are newer, and a library that lacks an entry point this module binds (built from older sources but stamped later, e.g. left
    over from another checkout) is rebuilt unconditionally.  A library that cannot be rebuilt is loaded as it is."""
    import subprocess
    try:
        subprocess.run(["make", "-s", "port"], cwd=_HERE, capture_output=True, check=False)
        nm = subprocess.run(["nm", "-D", "--defined-only", PORT_SO], capture_output=True, text=True, check=False)
    except OSError:
        return
    defined = {line.split()[-1] for line in nm.stdout.splitlines() if line.strip()}
    src = open(os.path.join(_HERE, "dab_oracle.h")).read()
    if nm.returncode == 0 and any(name not in defined for name in _declared(src)):
        subprocess.run(["make", "-s", "-B", "port"], cwd=_HERE, capture_output=True, check=False)


def _declared(header: str) -> List[str]:
    """the dabo_* functions oracle/dab_oracle.h declares"""
    import re
    return sorted(set(re.findall(r"\b(dabo_\w+)\s*\(", header)))


class PortLib:
    _inst = None

    @classmethod
    def get(cls) -> "PortLib":
        if cls._inst is None:
            cls._inst = cls()
        return cls._inst

    def __init__(self):
        _refresh_port()
        L = C.CDLL(PORT_SO)
        self.L = L
        L.dabo_pi_counts.argtypes = [C.c_int, _u8p]
        L.dabo_eep_segments.argtypes = [C.c_int, C.c_int, C.c_int, _i32p, _i32p]
        L.dabo_uep_segments.argtypes = [C.c_int, _i32p, _i32p]
        L.dabo_ofdm_params.argtypes = [C.c_int, _i32p]
        L.dabo_carrier_map.argtypes = [C.c_int, C.c_int, _i32p]
        L.dabo_prs_fft.argtypes = [C.c_int, _f32p, C.c_int]
        L.dabo_vit_decode.argtypes = [_i8p, C.c_int, _i32p, _i32p, C.c_int, _u8p, C.c_int, C.POINTER(C.c_uint64)]
        L.dabo_scrambler_bytes.argtypes = [_u8p, C.c_int]
        L.dabo_crc16.argtypes = [_u8p, C.c_int, C.c_uint16, C.c_uint16, C.c_uint16]
        L.dabo_crc16.restype = C.c_uint16
        L.dabo_fic_decode_group.argtypes = [_i8p, _u8p, _i32p]
        L.dabo_msc_create.argtypes = [C.c_int] * 6
        L.dabo_msc_create.restype = C.c_void_p
        L.dabo_msc_destroy.argtypes = [C.c_void_p]
        L.dabo_msc_decode_cif.argtypes = [C.c_void_p, _i8p, C.c_int, _u8p, C.c_int]
        L.dabo_rs_decode.argtypes = [C.c_int, C.c_int, _u8p, _i32p]
        L.dabo_aac_create.restype = C.c_void_p
        L.dabo_aac_destroy.argtypes = [C.c_void_p]
        L.dabo_aac_process.argtypes = [C.c_void_p, _u8p, C.c_int, _u8p, C.c_int]
        L.dabo_ofdm_create.argtypes = [C.c_int]
        L.dabo_ofdm_set_config.argtypes = [C.c_void_p, C.POINTER(OfdmConfig)]
        L.dabo_ofdm_create.restype = C.c_void_p
        L.dabo_ofdm_destroy.argtypes = [C.c_void_p]
        L.dabo_ofdm_frame_bits.argtypes = [C.c_void_p]
        L.dabo_ofdm_process_c32.argtypes = [C.c_void_p, _f32p, C.c_int]
        L.dabo_ofdm_process_u8.argtypes = [C.c_void_p, _u8p, C.c_int]
        L.dabo_ofdm_pop_frame.argtypes = [C.c_void_p, _i8p, _f32p, _i32p]
        L.dabo_ofdm_get_state.argtypes = [C.c_void_p, _i32p, _f32p]
        L.dabo_ofdm_keep_frames.argtypes = [C.c_void_p, C.c_int]
        L.dabo_fft.argtypes = [_f32p, C.c_int, C.c_int]
        L.dabo_time_ofdm_u8.argtypes = [C.c_int, _u8p, C.c_long, C.c_int, C.c_int, C.POINTER(C.c_int)]
        L.dabo_time_ofdm_u8.restype = C.c_double


class PortViterbi:
    def __init__(self):
        self.lib = PortLib.get().L

    def decode(self, soft: np.ndarray, segments: Sequence[Tuple[int, int]]) -> Tuple[np.ndarray, int, int]:
        soft = np.ascontiguousarray(soft, dtype=np.int8)
        pi, nb = _segs(segments)
        steps = int(nb.sum()) // 4
        n_out = (steps - 6) // 8
        out = np.zeros(n_out, dtype=np.uint8)
        err = C.c_uint64(0)
        consumed = self.lib.dabo_vit_decode(soft, soft.size, pi, nb, len(segments), out, n_out, C.byref(err))
        if consumed < 0:
            raise ValueError("dabo_vit_decode: bad arguments")
        return out, consumed, err.value


def port_scrambler_bytes(n: int) -> np.ndarray:
    out = np.zeros(n, dtype=np.uint8)
    PortLib.get().L.dabo_scrambler_bytes(out, n)
    return out


def port_segments(length=0, level=0, type_b=False, uep_index=None) -> List[Tuple[int, int]]:
    L = PortLib.get().L
    pi = np.zeros(5, dtype=np.int32)
    nb = np.zeros(5, dtype=np.int32)
    n = L.dabo_uep_segments(uep_index, pi, nb) if uep_index is not None else L.dabo_eep_segments(length, level, int(type_b), pi, nb)
    return [(int(pi[i]), int(nb[i])) for i in range(n)]


class PortFic:
    def __init__(self, nb_encoded_bits: int = 2304, nb_fibs_per_group: int = 3):
        self.lib = PortLib.get().L

    def decode_group_raw(self, bits: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
        bits = np.ascontiguousarray(bits, dtype=np.int8)
        out = np.zeros(96, dtype=np.uint8)
        ok = np.zeros(3, dtype=np.int32)
        self.lib.dabo_fic_decode_group(bits, out, ok)
        return out, ok

    def decode_group(self, bits: np.ndarray, cif_index: int = 0) -> List[bytes]:
        out, ok = self.decode_group_raw(bits)
        return [out[32 * i:32 * i + 30].tobytes() for i in range(3) if ok[i]]


class PortMsc:
    def __init__(self, start_address: int, length: int, is_uep: bool = False, uep_index: int = 0,
                 eep_level: int = 2, eep_type_b: bool = False):
        self.lib = PortLib.get().L
        self.h = self.lib.dabo_msc_create(start_address, length, int(is_uep), uep_index, eep_level, int(eep_type_b))
        self.cap = length * 8

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.dabo_msc_destroy(self.h)
            self.h = None

    def decode_cif(self, cif_bits: np.ndarray) -> np.ndarray:
        cif_bits = np.ascontiguousarray(cif_bits, dtype=np.int8)
        out = np.zeros(self.cap, dtype=np.uint8)
        n = self.lib.dabo_msc_decode_cif(self.h, cif_bits, cif_bits.size, out, self.cap)
        return out[:max(n, 0)].copy()


class PortRS:
    def __init__(self, nroots: int = 10, pad: int = 135):
        self.lib = PortLib.get().L
        self.nroots, self.pad = nroots, pad

    def decode(self, data: np.ndarray) -> Tuple[int, np.ndarray, np.ndarray]:
        d = np.ascontiguousarray(data, dtype=np.uint8).copy()
        pos = np.zeros(32, dtype=np.int32)
        cnt = self.lib.dabo_rs_decode(self.nroots, self.pad, d, pos)
        return cnt, d, pos[:max(cnt, 0)].copy()


class PortPacketFec:
    """Restatement of MSC_Reed_Solomon_Data_Packet_Processor (msc_reed_solomon_data_packet_processor.cpp:49-258) on top of the
    C restatement's RS decoder: a 2472-byte ring of whole packets, nine FEC packets with counters 0..8 close a set, the 12 rows
    of the 204-column table are decoded as RS(204,188) and only the application data table is corrected."""
    LENGTHS = (24, 48, 72, 96)
    RING = 2256 + 9 * 24

    def __init__(self):
        self.rs = PortRS(16, 51)
        self.ring = np.zeros(self.RING, dtype=np.uint8)
        self.rd = self.wr = self.fill = 0
        self.last = None

    def _pop(self):
        if self.fill == 0:
            return None
        n = self.LENGTHS[int(self.ring[self.rd]) >> 6]
        pkt = bytes(self.ring[(self.rd + np.arange(n)) % self.RING])
        self.fill -= n
        self.rd = (self.rd + n) % self.RING
        return pkt

    def _push(self, pkt: np.ndarray, lid: int):
        n = self.LENGTHS[lid]
        while self.RING - self.fill < n:                       # msc_reed_solomon_data_packet_processor.cpp:137-148
            m = self.LENGTHS[int(self.ring[self.rd]) >> 6]
            self.fill -= m
            self.rd = (self.rd + m) % self.RING
        idx = (self.wr + np.arange(n)) % self.RING
        self.ring[idx] = pkt[:n]
        self.ring[self.wr] = (int(pkt[0]) & 0x3F) | (lid << 6)    # :151-153 the length id is the one the processor decided on
        self.fill += n
        self.wr = (self.wr + n) % self.RING

    def _clear(self, out):
        while True:
            p = self._pop()
            if p is None:
                break
            out.append((p, False))

    def _correct(self, out):
        at = lambda off: (self.rd + off) % self.RING
        table = np.zeros(192, dtype=np.uint8)
        for i in range(9):                                     # :203-219
            n = 22 if i < 8 else 16
            table[22 * i:22 * i + n] = self.ring[[at(2256 + 24 * i + 2 + j) for j in range(n)]]
        for y in range(12):                                    # :222-258
            cw = np.concatenate([self.ring[[at(12 * x + y) for x in range(188)]], table[[12 * i + y for i in range(16)]]])
            cnt, fixed, pos = self.rs.decode(cw)
            if cnt < 0:
                continue
            for p in pos[:cnt]:
                x = int(p) - 51
                if 0 <= x < 188:
                    self.ring[at(12 * x + y)] = fixed[x]
        total = 0
        while total < 2256:
            p = self._pop()
            if p is None:
                break
            out.append((p, True))
            total += len(p)

    def read_packet(self, buf: np.ndarray) -> Tuple[int, List[Tuple[bytes, bool]]]:
        buf = np.asarray(buf, dtype=np.uint8)
        out: List[Tuple[bytes, bool]] = []
        if buf.size < 2:
            return int(buf.size), out
        lid = int(buf[0]) >> 6
        counter = (int(buf[0]) >> 2) & 0xF
        address = ((int(buf[0]) & 3) << 8) | int(buf[1])
        is_fec = address == 0x3FE
        if is_fec:
            lid = 0
        n = self.LENGTHS[lid]
        if buf.size < n:
            return int(buf.size), out
        self._push(buf, lid)
        if not is_fec:
            return n, out
        invalid = (counter != self.last + 1) if self.last is not None else (counter != 0)
        if invalid:
            self.last = None
            self._clear(out)
            return n, out
        self.last = counter
        if counter != 8:
            return n, out
        if self.fill != self.RING:
            self._clear(out)
        else:
            self._correct(out)
        self.last = None
        self.rd = self.wr = self.fill = 0
        return n, out


class PortAac:
    def __init__(self):
        self.lib = PortLib.get().L
        self.h = self.lib.dabo_aac_create()
        self.log = np.zeros(1 << 16, dtype=np.uint8)

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.dabo_aac_destroy(self.h)
            self.h = None

    def process(self, frame: np.ndarray) -> List[tuple]:
        frame = np.ascontiguousarray(frame, dtype=np.uint8)
        n = self.lib.dabo_aac_process(self.h, frame, frame.size, self.log, self.log.size)
        return parse_event_log(self.log[:n].tobytes())


class PortOfdm:
    def __init__(self, mode: int = 1, nb_threads: int = 1):
        self.lib = PortLib.get().L
        self.h = self.lib.dabo_ofdm_create(mode)
        if not self.h:
            raise ValueError(f"invalid transmission mode {mode}")
        self.frame_bits = self.lib.dabo_ofdm_frame_bits(self.h)
        self.config = dict(OFDM_DEFAULTS)

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.dabo_ofdm_destroy(self.h)
            self.h = None

    def set_config(self, **kw):
        """as RefOfdm.set_config"""
        self.config = _merge_config(self.config, kw)
        self.lib.dabo_ofdm_set_config(self.h, C.byref(OfdmConfig(**self.config)))

    def process_u8(self, iq_u8: np.ndarray, serial: bool = True):
        iq_u8 = np.ascontiguousarray(iq_u8, dtype=np.uint8)
        self.lib.dabo_ofdm_process_u8(self.h, iq_u8, iq_u8.size // 2)

    def process_c32(self, iq: np.ndarray, serial: bool = True):
        f = np.ascontiguousarray(iq, dtype=np.complex64).view(np.float32)
        self.lib.dabo_ofdm_process_c32(self.h, f, f.size // 2)

    def pop_frames(self):
        out = []
        while True:
            bits = np.zeros(self.frame_bits, dtype=np.int8)
            cf = np.zeros(2, dtype=np.float32)
            to = np.zeros(1, dtype=np.int32)
            if not self.lib.dabo_ofdm_pop_frame(self.h, bits, cf, to):
                break
            out.append((bits, float(cf[0]), float(cf[1]), int(to[0])))
        return out

    def state(self) -> dict:
        s = np.zeros(4, dtype=np.int32)
        f = np.zeros(3, dtype=np.float32)
        self.lib.dabo_ofdm_get_state(self.h, s, f)
        return dict(state=int(s[0]), frames_read=int(s[1]), frames_desync=int(s[2]), fine_time_offset=int(s[3]),
                    signal_avg=float(f[0]), coarse=float(f[1]), fine=float(f[2]))
