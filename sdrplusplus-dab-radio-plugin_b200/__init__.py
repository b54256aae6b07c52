"""B200-native DAB receive path: thin Python binding of the C ABI in include/dabgpu.h.

The product is csrc/libdabgpu.so (hand-written sm_100a kernels behind a C ABI).  This module only
loads it with ctypes for tests and bench.py; there is no Python or CPU implementation of the path
here, and loading fails loudly when the library has not been built.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libdabgpu.so")

OK, ERR_INVALID, ERR_CUDA, ERR_NOMEM, ERR_STATE, ERR_OVERFLOW = 0, -1, -2, -3, -4, -5
IQ_U8, IQ_C32 = 0, 1
MAX_SEGMENTS = 5
EV_FIRECODE_ERROR, EV_RS_ERROR, EV_SUPERFRAME_HEADER, EV_AU_CRC_ERROR, EV_ACCESS_UNIT = 1, 2, 3, 4, 5
WB_RAW_U8, WB_RAW_S8, WB_RAW_S16L, WB_RAW_F32L = 0, 1, 2, 3
WB_FORMATS = {"raw_u8": WB_RAW_U8, "raw_s8": WB_RAW_S8, "raw_s16l": WB_RAW_S16L, "raw_f32l": WB_RAW_F32L}
WB_BYTES_PER_SAMPLE = {WB_RAW_U8: 2, WB_RAW_S8: 2, WB_RAW_S16L: 4, WB_RAW_F32L: 8}


class DabGpuError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"dabgpu error {code}: {msg}")
        self.code = code


class OfdmConfig(C.Structure):
    _fields_ = [("signal_l1_update_beta", C.c_float), ("signal_l1_nb_samples", C.c_int), ("signal_l1_nb_decimate", C.c_int),
                ("null_thresh_start", C.c_float), ("null_thresh_end", C.c_float), ("fine_freq_update_beta", C.c_float),
                ("is_coarse_freq_correction", C.c_int), ("max_coarse_freq_correction_norm", C.c_float),
                ("coarse_freq_slow_beta", C.c_float), ("impulse_peak_threshold_db", C.c_float),
                ("impulse_peak_distance_probability", C.c_float)]


class Config(C.Structure):
    _fields_ = [("device", C.c_int), ("transmission_mode", C.c_int), ("max_streams", C.c_int), ("iq_format", C.c_int),
                ("ring_samples", C.c_size_t), ("frame_slots", C.c_int), ("max_subchannels", C.c_int),
                ("cuda_stream", C.c_void_p), ("ofdm", OfdmConfig), ("flags", C.c_uint)]


class Params(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("nb_frame_symbols", "nb_symbol_period", "nb_null_period", "nb_cyclic_prefix", "nb_fft",
                                       "nb_data_carriers", "nb_frame_bits", "nb_fic_bits", "nb_msc_bits", "nb_cifs",
                                       "nb_fibs_per_cif", "nb_fib_group_bits", "nb_cif_bits", "nb_frame_samples")]


class OfdmStatus(C.Structure):
    _fields_ = [("state", C.c_int), ("total_frames_read", C.c_int), ("total_frames_desync", C.c_int), ("fine_time_offset", C.c_int),
                ("signal_l1_average", C.c_float), ("freq_coarse_offset", C.c_float), ("freq_fine_offset", C.c_float),
                ("frames_queued", C.c_int), ("frames_dropped", C.c_int)]


class FrameInfo(C.Structure):
    _fields_ = [("freq_coarse_offset", C.c_float), ("freq_fine_offset", C.c_float), ("fine_time_offset", C.c_int), ("frame_index", C.c_int)]


class ViterbiJob(C.Structure):
    _fields_ = [("soft_offset", C.c_uint64), ("n_soft", C.c_uint32), ("n_seg", C.c_uint32), ("seg_pi", C.c_uint8 * (MAX_SEGMENTS + 3)),
                ("seg_bits", C.c_uint32 * MAX_SEGMENTS), ("out_offset", C.c_uint64), ("n_out_bytes", C.c_uint32), ("descramble", C.c_uint32)]


class SubchannelC(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("start_address", "length", "is_uep", "uep_prot_index", "eep_prot_level", "eep_type_b", "is_dabplus")]


class ChanStatus(C.Structure):
    _fields_ = [("decoded", C.c_int), ("frame_index", C.c_int)]


class Counters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("frames_demodulated", "frames_channel_decoded", "fibs_crc_ok", "fibs_total", "msc_bytes_decoded",
                                          "superframes_ok", "superframes_rs_fail", "superframes_firecode_fail", "au_ok", "au_crc_fail",
                                          "frames_dropped")]


class Profile(C.Structure):
    _fields_ = [("ms", C.c_double * 5), ("launches", C.c_uint64 * 5)]


class Step(C.Structure):
    """dabgpu_step (include/dabgpu.h): one pipelined push of IQ with optional result pointers."""
    _fields_ = [("iq_host", C.c_void_p), ("iq_stride_bytes", C.c_size_t), ("first_stream", C.c_int), ("n_streams", C.c_int),
                ("n_samples", C.c_int), ("block_size", C.c_int), ("run_chan_decode", C.c_int), ("frames_host", C.c_void_p),
                ("produced_host", C.c_void_p), ("msc_host", C.c_void_p), ("msc_valid_host", C.c_void_p), ("fic_host", C.c_void_p),
                ("fic_crc_host", C.c_void_p), ("chan_status_host", C.c_void_p)]


class WidebandConfig(C.Structure):
    _fields_ = [("sample_rate", C.c_int), ("format", C.c_int), ("n_sources", C.c_int), ("n_channels", C.c_int),
                ("source", C.POINTER(C.c_int)), ("offset_hz", C.POINTER(C.c_int))]


class WidebandGeometry(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("bin_hz", "fft_in", "fft_out", "step_in", "step_out", "taps")]


CIF_OUT_STRIDE, FIC_GROUP_STRIDE, PIPELINE_DEPTH = 6912, 128, 2

PROF_CLASSES = ("ofdm_ctl", "ofdm_demod", "viterbi", "dabplus", "chan_misc")

EXPORTS = [
    "dabgpu_profile_enable", "dabgpu_profile_read",
    "dabgpu_version", "dabgpu_last_error", "dabgpu_device_count", "dabgpu_config_default", "dabgpu_ctx_create", "dabgpu_ctx_destroy",
    "dabgpu_sync", "dabgpu_cuda_stream", "dabgpu_launch_count", "dabgpu_get_params", "dabgpu_ofdm_reset", "dabgpu_ofdm_process",
    "dabgpu_ofdm_attach_device_input", "dabgpu_ofdm_advance", "dabgpu_ofdm_get_status", "dabgpu_ofdm_pop_frames",
    "dabgpu_ofdm_fetch_latest", "dabgpu_viterbi_decode", "dabgpu_msc_configure", "dabgpu_softbits_push", "dabgpu_chan_decode",
    "dabgpu_chan_get_status", "dabgpu_chan_get_fic", "dabgpu_chan_get_msc", "dabgpu_chan_get_dabplus_events", "dabgpu_rs_decode",
    "dabgpu_get_counters", "dabgpu_submit", "dabgpu_wait", "dabgpu_msc_get_layout",
    "dabgpu_ofdm_set_config", "dabgpu_fic_decode", "dabgpu_dabplus_open", "dabgpu_dabplus_close", "dabgpu_dabplus_process",
    "dabgpu_autocfg_create", "dabgpu_autocfg_destroy", "dabgpu_autocfg_push_fibs", "dabgpu_autocfg_dump", "dabgpu_autocfg_runnable",
    "dabgpu_host_alloc", "dabgpu_host_free", "dabgpu_ofdm_get_frame_data_vec", "dabgpu_ofdm_get_correlation_buffer", "dabgpu_autocfg_applied", "dabgpu_msc_add_subchannel", "dabgpu_msc_remove_subchannel", "dabgpu_chan_join",
    "dabgpu_autocfg_apply", "dabgpu_ofdm_get_response", "dabgpu_ofdm_get_frame_fft", "dabgpu_iq_convert", "dabgpu_softbits_to_bytes", "dabgpu_bytes_to_softbits",
    "dabgpu_packet_fec_decode", "dabgpu_wideband_open", "dabgpu_wideband_process", "dabgpu_wideband_close",
    "dabgpu_wideband_plan", "dabgpu_wideband_open_any_rate", "dabgpu_wideband_reserve", "dabgpu_wideband_submit",
]

_lib = None


def load_library() -> C.CDLL:
    """Loads csrc/libdabgpu.so.  Raises if it was not built: there is no fallback implementation."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DabGpuError(ERR_STATE, f"{LIB_PATH} is missing: run __graft_entry__.build() (nvcc, sm_100a). No CPU fallback exists.")
    L = C.CDLL(LIB_PATH)
    L.dabgpu_version.restype = C.c_char_p
    L.dabgpu_last_error.restype = C.c_char_p
    L.dabgpu_config_default.argtypes = [C.POINTER(Config), C.c_int]
    L.dabgpu_config_default.restype = None
    L.dabgpu_ctx_create.argtypes = [C.POINTER(Config), C.POINTER(C.c_void_p)]
    L.dabgpu_ctx_destroy.argtypes = [C.c_void_p]
    L.dabgpu_ctx_destroy.restype = None
    L.dabgpu_sync.argtypes = [C.c_void_p]
    L.dabgpu_host_alloc.argtypes = [C.POINTER(C.c_void_p), C.c_size_t, C.c_int]
    L.dabgpu_host_free.argtypes = [C.c_void_p]
    L.dabgpu_host_free.restype = None
    L.dabgpu_cuda_stream.argtypes = [C.c_void_p]
    L.dabgpu_cuda_stream.restype = C.c_void_p
    L.dabgpu_launch_count.argtypes = [C.c_void_p]
    L.dabgpu_launch_count.restype = C.c_uint64
    L.dabgpu_get_params.argtypes = [C.c_int, C.POINTER(Params)]
    L.dabgpu_profile_enable.argtypes = [C.c_void_p, C.c_int]
    L.dabgpu_profile_read.argtypes = [C.c_void_p, C.POINTER(Profile)]
    L.dabgpu_ofdm_reset.argtypes = [C.c_void_p, C.c_int]
    L.dabgpu_ofdm_process.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int]
    L.dabgpu_ofdm_attach_device_input.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t]
    L.dabgpu_ofdm_advance.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]
    L.dabgpu_ofdm_get_status.argtypes = [C.c_void_p, C.c_int, C.POINTER(OfdmStatus)]
    L.dabgpu_ofdm_pop_frames.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.POINTER(FrameInfo), C.POINTER(C.c_int)]
    L.dabgpu_ofdm_fetch_latest.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.dabgpu_viterbi_decode.argtypes = [C.c_void_p, C.POINTER(ViterbiJob), C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]
    L.dabgpu_msc_configure.argtypes = [C.c_void_p, C.c_int, C.POINTER(SubchannelC), C.c_int]
    L.dabgpu_msc_add_subchannel.argtypes = [C.c_void_p, C.c_int, C.POINTER(SubchannelC), C.POINTER(C.c_int)]
    L.dabgpu_msc_remove_subchannel.argtypes = [C.c_void_p, C.c_int, C.c_int]
    L.dabgpu_chan_join.argtypes = [C.c_void_p]
    L.dabgpu_softbits_push.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int]
    L.dabgpu_chan_decode.argtypes = [C.c_void_p, C.c_int, C.c_int]
    L.dabgpu_chan_get_status.argtypes = [C.c_void_p, C.c_int, C.POINTER(ChanStatus)]
    L.dabgpu_chan_get_fic.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.dabgpu_chan_get_msc.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.POINTER(C.c_int)]
    L.dabgpu_chan_get_dabplus_events.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
    L.dabgpu_rs_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.dabgpu_packet_fec_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    L.dabgpu_get_counters.argtypes = [C.c_void_p, C.POINTER(Counters)]
    L.dabgpu_ofdm_set_config.argtypes = [C.c_void_p, C.POINTER(OfdmConfig)]
    L.dabgpu_fic_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.dabgpu_dabplus_open.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    L.dabgpu_dabplus_close.argtypes = [C.c_void_p, C.c_void_p]
    L.dabgpu_dabplus_close.restype = None
    L.dabgpu_dabplus_process.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
    L.dabgpu_submit.argtypes = [C.c_void_p, C.POINTER(Step), C.POINTER(C.c_uint64)]
    L.dabgpu_wait.argtypes = [C.c_void_p, C.c_uint64]
    L.dabgpu_msc_get_layout.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.dabgpu_autocfg_create.restype = C.c_void_p
    L.dabgpu_autocfg_destroy.argtypes = [C.c_void_p]
    L.dabgpu_autocfg_destroy.restype = None
    L.dabgpu_autocfg_push_fibs.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_void_p]
    L.dabgpu_autocfg_dump.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int), C.c_void_p, C.c_int, C.POINTER(C.c_int)]
    L.dabgpu_autocfg_runnable.argtypes = [C.c_void_p, C.POINTER(SubchannelC), C.c_void_p, C.c_int, C.POINTER(C.c_int)]
    L.dabgpu_autocfg_apply.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    L.dabgpu_autocfg_applied.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
    L.dabgpu_ofdm_get_response.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int]
    L.dabgpu_ofdm_get_frame_fft.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]
    L.dabgpu_ofdm_get_frame_data_vec.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]
    L.dabgpu_ofdm_get_correlation_buffer.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]
    L.dabgpu_iq_convert.argtypes = [C.c_char_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
    L.dabgpu_softbits_to_bytes.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p]
    L.dabgpu_bytes_to_softbits.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p]
    L.dabgpu_wideband_open.argtypes = [C.c_void_p, C.POINTER(WidebandConfig), C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]
    L.dabgpu_wideband_process.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_int, C.POINTER(C.c_size_t)]
    L.dabgpu_wideband_close.argtypes = [C.c_void_p]
    L.dabgpu_wideband_plan.argtypes = [C.c_int, C.POINTER(WidebandGeometry)]
    L.dabgpu_wideband_open_any_rate.argtypes = L.dabgpu_wideband_open.argtypes
    L.dabgpu_wideband_reserve.argtypes = [C.c_void_p, C.c_size_t]
    L.dabgpu_wideband_submit.argtypes = [C.c_void_p, C.POINTER(Step), C.POINTER(C.c_uint64)]
    _lib = L
    return L


def _check(rc: int):
    if rc != OK:
        raise DabGpuError(rc, load_library().dabgpu_last_error().decode(errors="replace"))


class HostBuffer:
    """Page-locked host memory from dabgpu_host_alloc, viewed as a numpy uint8 array (`.array`)."""

    def __init__(self, nbytes: int, write_combined: bool = False):
        self.L = load_library()
        self.ptr = C.c_void_p()
        _check(self.L.dabgpu_host_alloc(C.byref(self.ptr), nbytes, int(write_combined)))
        self.nbytes = nbytes
        self.array = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(self.ptr.value))

    def close(self):
        if getattr(self, "ptr", None) and self.ptr.value:
            self.array = None
            self.L.dabgpu_host_free(self.ptr)
            self.ptr = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def get_params(mode: int) -> Params:
    p = Params()
    _check(load_library().dabgpu_get_params(mode, C.byref(p)))
    return p


def wideband_plan(rate: int) -> dict:
    """dabgpu_wideband_plan: the wideband filter bank's block geometry at `rate` Hz (bin_hz, fft_in, fft_out, step_in, step_out,
    taps); raises DabGpuError for a rate it does not support.  Needs no GPU."""
    g = WidebandGeometry()
    _check(load_library().dabgpu_wideband_plan(rate, C.byref(g)))
    return {n: getattr(g, n) for n, _ in WidebandGeometry._fields_}


def _ptr(a: np.ndarray) -> C.c_void_p:
    return C.c_void_p(a.ctypes.data)


def _step(iq_ptr, iq_stride_bytes, n_samples, block_size, first_stream, n_streams, run_chan_decode, out_ptrs) -> Step:
    st = Step()
    st.iq_host, st.iq_stride_bytes = iq_ptr, iq_stride_bytes
    st.first_stream, st.n_streams = first_stream, n_streams
    st.n_samples, st.block_size, st.run_chan_decode = n_samples, block_size, int(run_chan_decode)
    for k, v in out_ptrs.items():
        setattr(st, k, v)
    return st


class DabGpu:
    """One context = one GPU, `max_streams` independent IQ streams (mirrors Radio_Block x N)."""

    def __init__(self, mode: int = 1, max_streams: int = 1, device: int = 0, iq_format: int = IQ_U8, ring_samples: int = 0,
                 frame_slots: int = 0, max_subchannels: int = 0, cuda_stream: Optional[int] = None, ofdm_overrides: Optional[dict] = None,
                 flags: int = 0):
        self.L = load_library()
        cfg = Config()
        self.L.dabgpu_config_default(C.byref(cfg), mode)
        cfg.device = device
        cfg.max_streams = max_streams
        cfg.iq_format = iq_format
        cfg.ring_samples = ring_samples
        cfg.frame_slots = frame_slots
        cfg.max_subchannels = max_subchannels
        cfg.cuda_stream = cuda_stream
        cfg.flags = flags
        self._ofdm_cfg = dict(ofdm_overrides or {})
        for k, v in (ofdm_overrides or {}).items():
            setattr(cfg.ofdm, k, v)
        self.h = C.c_void_p()
        _check(self.L.dabgpu_ctx_create(C.byref(cfg), C.byref(self.h)))
        self.mode = mode
        self.max_streams = max_streams
        self.iq_format = iq_format
        self.P = get_params(mode)
        self._subs = {}

    def close(self):
        if getattr(self, "_wideband", None) is not None:
            self._wideband.close()
        if getattr(self, "h", None):
            self.L.dabgpu_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        _check(self.L.dabgpu_sync(self.h))

    @property
    def cuda_stream(self) -> int:
        return int(self.L.dabgpu_cuda_stream(self.h) or 0)

    @property
    def launch_count(self) -> int:
        return int(self.L.dabgpu_launch_count(self.h))

    def profile_enable(self, on: bool = True):
        _check(self.L.dabgpu_profile_enable(self.h, int(on)))

    def profile_read(self) -> dict:
        p = Profile()
        _check(self.L.dabgpu_profile_read(self.h, C.byref(p)))
        return {name: {"ms": p.ms[i], "launches": int(p.launches[i])} for i, name in enumerate(PROF_CLASSES)}

    # ---- Viterbi -------------------------------------------------------------------------
    def viterbi_decode(self, soft_list: Sequence[np.ndarray], segments_list: Sequence[Sequence[Tuple[int, int]]],
                       descramble: bool = False, n_out_bytes: Optional[Sequence[int]] = None):
        """Batch of independent trellises.  Returns (list of byte arrays, path errors)."""
        n = len(soft_list)
        jobs = (ViterbiJob * n)()
        soft_off, out_off = 0, 0
        outs = []
        for i, (soft, segs) in enumerate(zip(soft_list, segments_list)):
            steps = sum(nb for _, nb in segs) // 4
            nout = (steps - 6) // 8 if n_out_bytes is None else n_out_bytes[i]
            j = jobs[i]
            j.soft_offset, j.n_soft, j.n_seg = soft_off, soft.size, len(segs)
            for k, (pi, nb) in enumerate(segs):
                j.seg_pi[k] = pi
                j.seg_bits[k] = nb
            j.out_offset, j.n_out_bytes, j.descramble = out_off, nout, int(descramble)
            soft_off += soft.size
            outs.append((out_off, nout))
            out_off += (nout + 15) & ~15
        soft_all = np.ascontiguousarray(np.concatenate([np.asarray(s, dtype=np.int8) for s in soft_list]))
        out = np.zeros(max(out_off, 16), dtype=np.uint8)
        perr = np.zeros(n, dtype=np.uint64)
        _check(self.L.dabgpu_viterbi_decode(self.h, jobs, n, _ptr(soft_all), soft_all.size, _ptr(out), out.size, _ptr(perr)))
        return [out[o:o + m].copy() for o, m in outs], perr

    # ---- channel decode ------------------------------------------------------------------
    @staticmethod
    def _fill_sub(dst: SubchannelC, s) -> None:
        dst.start_address, dst.length = s.start_address, s.length
        dst.is_uep, dst.uep_prot_index = int(s.is_uep), s.uep_index
        dst.eep_prot_level, dst.eep_type_b = s.eep_level, int(s.eep_type_b)
        dst.is_dabplus = int(getattr(s, "dabplus", False))

    def msc_configure(self, stream: int, subs: Sequence) -> None:
        arr = (SubchannelC * max(len(subs), 1))()
        for i, s in enumerate(subs):
            self._fill_sub(arr[i], s)
        _check(self.L.dabgpu_msc_configure(self.h, stream, arr, len(subs)))
        self._subs[stream] = list(subs)

    def msc_add_subchannel(self, stream: int, sub) -> int:
        """Attach one more decoder without touching the running ones; returns its sub_index."""
        d = SubchannelC()
        self._fill_sub(d, sub)
        idx = C.c_int(-1)
        _check(self.L.dabgpu_msc_add_subchannel(self.h, stream, C.byref(d), C.byref(idx)))
        self._subs.setdefault(stream, []).append(sub)
        return idx.value

    def msc_remove_subchannel(self, stream: int, sub_index: int) -> None:
        _check(self.L.dabgpu_msc_remove_subchannel(self.h, stream, sub_index))

    def chan_join(self) -> None:
        """Non-blocking: work queued on the context's stream from now on waits for the last chan_decode."""
        _check(self.L.dabgpu_chan_join(self.h))

    def softbits_push(self, frames: np.ndarray, first_stream: int = 0) -> None:
        """frames: [n_streams, nb_frame_bits] int8"""
        frames = np.ascontiguousarray(frames, dtype=np.int8)
        assert frames.ndim == 2 and frames.shape[1] == self.P.nb_frame_bits
        _check(self.L.dabgpu_softbits_push(self.h, _ptr(frames), frames.shape[1], first_stream, frames.shape[0]))

    def chan_decode(self, first_stream: int = 0, n_streams: Optional[int] = None) -> None:
        _check(self.L.dabgpu_chan_decode(self.h, first_stream, self.max_streams - first_stream if n_streams is None else n_streams))

    def chan_status(self, stream: int) -> Tuple[int, int]:
        st = ChanStatus()
        _check(self.L.dabgpu_chan_get_status(self.h, stream, C.byref(st)))
        return st.decoded, st.frame_index

    def get_fic(self, stream: int) -> Tuple[np.ndarray, np.ndarray]:
        n = self.P.nb_cifs * self.P.nb_fibs_per_cif
        fibs = np.zeros((n, 32), dtype=np.uint8)
        ok = np.zeros(n, dtype=np.uint8)
        _check(self.L.dabgpu_chan_get_fic(self.h, stream, _ptr(fibs), _ptr(ok)))
        return fibs, ok

    def get_msc(self, stream: int, sub_index: int) -> Tuple[np.ndarray, np.ndarray]:
        nb = C.c_int(0)
        _check(self.L.dabgpu_chan_get_msc(self.h, stream, sub_index, None, 0, None, C.byref(nb)))
        out = np.zeros((self.P.nb_cifs, nb.value), dtype=np.uint8)
        valid = np.zeros(self.P.nb_cifs, dtype=np.uint8)
        _check(self.L.dabgpu_chan_get_msc(self.h, stream, sub_index, _ptr(out), out.size, _ptr(valid), C.byref(nb)))
        return out, valid

    def get_dabplus_events(self, stream: int, sub_index: int) -> bytes:
        buf = np.zeros(1 << 16, dtype=np.uint8)
        n = C.c_size_t(0)
        _check(self.L.dabgpu_chan_get_dabplus_events(self.h, stream, sub_index, _ptr(buf), buf.size, C.byref(n)))
        return buf[:n.value].tobytes()

    def rs_decode(self, codewords: np.ndarray, nroots: int = 10, pad: int = 135):
        cw = np.ascontiguousarray(codewords, dtype=np.uint8).copy()
        assert cw.ndim == 2 and cw.shape[1] == 255 - pad
        counts = np.zeros(cw.shape[0], dtype=np.int32)
        pos = np.zeros((cw.shape[0], nroots), dtype=np.int32)
        _check(self.L.dabgpu_rs_decode(self.h, _ptr(cw), cw.shape[0], nroots, pad, _ptr(counts), _ptr(pos)))
        return counts, cw, pos

    def packet_fec_decode(self, frames: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
        """frames [n][2448] (application data table + RS data table, transport order) -> (corrected frames, row counts [n][12])"""
        fr = np.ascontiguousarray(frames, dtype=np.uint8).copy()
        assert fr.ndim == 2 and fr.shape[1] == 2448
        counts = np.zeros((fr.shape[0], 12), dtype=np.int32)
        _check(self.L.dabgpu_packet_fec_decode(self.h, _ptr(fr), fr.shape[0], _ptr(counts)))
        return fr, counts

    def fic_decode(self, soft: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
        """soft: [n_groups, 2304] int8 -> (fibs [n_groups, 3, 32], crc_ok [n_groups, 3])"""
        soft = np.ascontiguousarray(soft, dtype=np.int8).reshape(-1, 2304)
        fibs = np.zeros((soft.shape[0], 3, 32), dtype=np.uint8)
        ok = np.zeros((soft.shape[0], 3), dtype=np.uint8)
        _check(self.L.dabgpu_fic_decode(self.h, _ptr(soft), soft.shape[0], _ptr(fibs), _ptr(ok)))
        return fibs, ok

    def dabplus_open(self) -> int:
        h = C.c_void_p()
        _check(self.L.dabgpu_dabplus_open(self.h, C.byref(h)))
        return h.value

    def dabplus_close(self, proc: int) -> None:
        self.L.dabgpu_dabplus_close(self.h, C.c_void_p(proc))

    def dabplus_process(self, proc: int, frame: np.ndarray) -> bytes:
        frame = np.ascontiguousarray(frame, dtype=np.uint8)
        buf = np.zeros(1 << 16, dtype=np.uint8)
        n = C.c_size_t(0)
        _check(self.L.dabgpu_dabplus_process(self.h, C.c_void_p(proc), _ptr(frame), frame.size, _ptr(buf), buf.size, C.byref(n)))
        return buf[:n.value].tobytes()

    def ofdm_set_config(self, **kw) -> None:
        cfg = Config()
        self.L.dabgpu_config_default(C.byref(cfg), self.mode)
        for k, v in {**getattr(self, "_ofdm_cfg", {}), **kw}.items():
            setattr(cfg.ofdm, k, v)
        self._ofdm_cfg = {**getattr(self, "_ofdm_cfg", {}), **kw}
        _check(self.L.dabgpu_ofdm_set_config(self.h, C.byref(cfg.ofdm)))

    def counters(self) -> dict:
        c = Counters()
        _check(self.L.dabgpu_get_counters(self.h, C.byref(c)))
        return {n: int(getattr(c, n)) for n, _ in Counters._fields_}

    # ---- OFDM ----------------------------------------------------------------------------
    def ofdm_reset(self, stream: int = -1):
        _check(self.L.dabgpu_ofdm_reset(self.h, stream))

    def ofdm_process(self, iq: np.ndarray, first_stream: int = 0, block_size: int = 65536):
        """iq: [n_streams, n_samples*2] uint8 (IQ_U8) or [n_streams, n_samples] complex64 (IQ_C32), host memory."""
        if self.iq_format == IQ_U8:
            iq = np.ascontiguousarray(iq, dtype=np.uint8)
            n_samples = iq.shape[1] // 2
        else:
            iq = np.ascontiguousarray(iq, dtype=np.complex64)
            n_samples = iq.shape[1]
        _check(self.L.dabgpu_ofdm_process(self.h, _ptr(iq), iq.strides[0], first_stream, iq.shape[0], n_samples, block_size))

    def ofdm_attach_device_input(self, dev_ptr: int, stream_stride_samples: int, capacity_samples: int):
        _check(self.L.dabgpu_ofdm_attach_device_input(self.h, C.c_void_p(dev_ptr), stream_stride_samples, capacity_samples))

    def ofdm_advance(self, n_samples: int, block_size: int = 65536, first_stream: int = 0, n_streams: Optional[int] = None):
        _check(self.L.dabgpu_ofdm_advance(self.h, first_stream, self.max_streams - first_stream if n_streams is None else n_streams,
                                          n_samples, block_size))

    def wideband_open(self, sample_rate: int, fmt, sources: Sequence[int], offsets_hz: Sequence[int], d_out: int,
                      capacity_samples: int, n_sources: Optional[int] = None, any_rate: bool = False) -> "Wideband":
        """dabgpu_wideband_open: channel c = ensemble of capture sources[c] at offsets_hz[c] from its centre, written as c32 to the
        device buffer d_out ([channel][capacity_samples], e.g. a torch.complex64 tensor's data_ptr()) and fed to stream c.
        any_rate=True: dabgpu_wideband_open_any_rate, which takes every rate wideband_plan() supports."""
        w = Wideband(self, sample_rate, fmt, sources, offsets_hz, d_out, capacity_samples, n_sources, any_rate)
        self._wideband = w
        return w

    def submit(self, iq_ptr: int, iq_stride_bytes: int, n_samples: int, block_size: int = 65536, first_stream: int = 0,
               n_streams: Optional[int] = None, run_chan_decode: bool = False, **out_ptrs) -> int:
        """dabgpu_submit: queue H2D + OFDM (+ channel decode) + D2H without blocking; returns the ticket.
        out_ptrs: frames_host, produced_host, msc_host, msc_valid_host, fic_host, fic_crc_host, chan_status_host (raw addresses)."""
        st = _step(iq_ptr, iq_stride_bytes, n_samples, block_size, first_stream,
                   self.max_streams - first_stream if n_streams is None else n_streams, run_chan_decode, out_ptrs)
        t = C.c_uint64(0)
        _check(self.L.dabgpu_submit(self.h, C.byref(st), C.byref(t)))
        return int(t.value)

    def wait(self, ticket: int) -> None:
        _check(self.L.dabgpu_wait(self.h, ticket))

    def msc_layout(self, stream: int, sub_index: int) -> Tuple[int, int]:
        off, nb = C.c_int(0), C.c_int(0)
        _check(self.L.dabgpu_msc_get_layout(self.h, stream, sub_index, C.byref(off), C.byref(nb)))
        return off.value, nb.value

    def ofdm_status(self, stream: int) -> dict:
        st = OfdmStatus()
        _check(self.L.dabgpu_ofdm_get_status(self.h, stream, C.byref(st)))
        return {n: getattr(st, n) for n, _ in OfdmStatus._fields_}

    def ofdm_response(self, stream: int, kind: int) -> np.ndarray:
        """GUI tap: kind 0 = impulse response, 1 = coarse frequency response (dB, nb_fft floats); needs FLAG_DIAG_TAPS."""
        out = np.empty(self.P.nb_fft, dtype=np.float32)
        _check(self.L.dabgpu_ofdm_get_response(self.h, stream, kind, out.ctypes.data, out.size))
        return out

    def ofdm_frame_fft(self, stream: int, with_null: bool = False) -> np.ndarray:
        """GUI tap: (nb_frame_symbols [+ 1 NULL row], nb_fft) complex64 spectra of the last emitted frame; needs FLAG_DIAG_TAPS."""
        out = np.empty((self.P.nb_frame_symbols + int(with_null), self.P.nb_fft), dtype=np.complex64)
        _check(self.L.dabgpu_ofdm_get_frame_fft(self.h, stream, out.ctypes.data, out.size * 2))
        return out

    def ofdm_correlation_buffer(self, stream: int) -> np.ndarray:
        """GUI tap: the NULL + PRS correlation window, nb_null_period + nb_symbol_period complex64."""
        out = np.empty(self.P.nb_null_period + self.P.nb_symbol_period, dtype=np.complex64)
        _check(self.L.dabgpu_ofdm_get_correlation_buffer(self.h, stream, out.ctypes.data, out.size * 2))
        return out

    def ofdm_frame_data_vec(self, stream: int) -> np.ndarray:
        """GUI tap: (nb_frame_symbols - 1, nb_data_carriers) complex64 DQPSK vectors of the last emitted frame."""
        out = np.empty((self.P.nb_frame_symbols - 1, self.P.nb_data_carriers), dtype=np.complex64)
        _check(self.L.dabgpu_ofdm_get_frame_data_vec(self.h, stream, out.ctypes.data, out.size * 2))
        return out

    def ofdm_pop_frames(self, stream: int, max_frames: int = 64):
        frames = np.zeros((max_frames, self.P.nb_frame_bits), dtype=np.int8)
        infos = (FrameInfo * max_frames)()
        n = C.c_int(0)
        _check(self.L.dabgpu_ofdm_pop_frames(self.h, stream, _ptr(frames), max_frames, infos, C.byref(n)))
        return [(frames[i].copy(), infos[i].freq_coarse_offset, infos[i].freq_fine_offset, infos[i].fine_time_offset) for i in range(n.value)]

    def ofdm_fetch_latest(self, first_stream: int = 0, n_streams: Optional[int] = None):
        n = self.max_streams - first_stream if n_streams is None else n_streams
        frames = np.zeros((n, self.P.nb_frame_bits), dtype=np.int8)
        produced = np.zeros(n, dtype=np.uint8)
        _check(self.L.dabgpu_ofdm_fetch_latest(self.h, first_stream, n, _ptr(frames), _ptr(produced)))
        return frames, produced


class Wideband:
    """Wideband front end of one context (dabgpu_wideband_*): splits multi-ensemble captures into the context's streams."""

    def __init__(self, ctx: DabGpu, sample_rate: int, fmt, sources: Sequence[int], offsets_hz: Sequence[int], d_out: int,
                 capacity_samples: int, n_sources: Optional[int] = None, any_rate: bool = False):
        self.L, self.ctx = ctx.L, ctx
        self.format = WB_FORMATS[fmt] if isinstance(fmt, str) else int(fmt)
        self.n_sources = (max(sources) + 1 if len(sources) else 0) if n_sources is None else n_sources
        self.n_channels = len(sources)
        src = (C.c_int * max(len(sources), 1))(*sources)
        off = (C.c_int * max(len(offsets_hz), 1))(*offsets_hz)
        cfg = WidebandConfig(sample_rate, self.format, self.n_sources, len(sources), src, off)
        self.h = C.c_void_p()
        fn = self.L.dabgpu_wideband_open_any_rate if any_rate else self.L.dabgpu_wideband_open
        _check(fn(ctx.h, C.byref(cfg), C.c_void_p(d_out), capacity_samples, C.byref(self.h)))

    def process(self, iq: np.ndarray, block_size: int = 65536) -> int:
        """iq: [n_sources, ...] host array, each row one source's raw samples (u8 / s8 / s16 I,Q pairs, f32 I,Q or complex64).
        Returns the new output samples per channel."""
        assert iq.ndim == 2 and iq.shape[0] == self.n_sources and iq.strides[1] == iq.itemsize
        n = (iq.shape[1] * iq.itemsize) // WB_BYTES_PER_SAMPLE[self.format]
        n_out = C.c_size_t(0)
        _check(self.L.dabgpu_wideband_process(self.h, C.c_void_p(iq.ctypes.data), iq.strides[0], n, block_size, C.byref(n_out)))
        return n_out.value

    def reserve(self, max_samples: int) -> None:
        """dabgpu_wideband_reserve: size the input ring for submit() tickets of up to max_samples raw samples per source.
        Only before the first input."""
        _check(self.L.dabgpu_wideband_reserve(self.h, max_samples))

    def submit(self, iq_ptr: int, source_stride_bytes: int, n_samples: int, block_size: int = 65536, first_stream: int = 0,
               n_streams: Optional[int] = None, run_chan_decode: bool = False, **out_ptrs) -> int:
        """dabgpu_wideband_submit: queue the upload of n_samples raw samples per source (source s at iq_ptr + s *
        source_stride_bytes, pinned host memory that stays valid until the ticket is waited for), the filter bank and OFDM over
        every channel, the channel decode of channels [first_stream, first_stream + n_streams) if run_chan_decode, and the
        copy-out of out_ptrs (as DabGpu.submit, rows from first_stream) without blocking.  Returns the ticket; retire it with
        DabGpu.wait."""
        st = _step(iq_ptr, source_stride_bytes, n_samples, block_size, first_stream,
                   self.n_channels - first_stream if n_streams is None else n_streams, run_chan_decode, out_ptrs)
        t = C.c_uint64(0)
        _check(self.L.dabgpu_wideband_submit(self.h, C.byref(st), C.byref(t)))
        return int(t.value)

    def close(self):
        if getattr(self, "h", None):
            self.L.dabgpu_wideband_close(self.h)
            self.h = None
            if getattr(self.ctx, "_wideband", None) is self:
                self.ctx._wideband = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class FicAutoConfig:
    """Self-configuration from the FIC (host only): FIBs in, sub-channel table out (dabgpu_autocfg_*, include/dabgpu.h).
    Mirrors FIG_Processor -> Radio_FIG_Handler -> DAB_Database_Updater -> BasicRadio::UpdateAfterProcessing of the reference
    for FIG 0/1, 0/2, 0/3 and 0/14."""

    def __init__(self):
        self.L = load_library()
        self.h = C.c_void_p(self.L.dabgpu_autocfg_create())

    def close(self):
        if self.h:
            self.L.dabgpu_autocfg_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def push_fibs(self, fibs: np.ndarray, crc_ok: Optional[np.ndarray] = None) -> int:
        """fibs: (n, >=30) uint8 rows.  Returns how many of them changed the database."""
        fibs = np.ascontiguousarray(fibs, dtype=np.uint8)
        if fibs.ndim == 1:
            fibs = fibs.reshape(1, -1)
        ok = None if crc_ok is None else np.ascontiguousarray(crc_ok, dtype=np.uint8)
        rc = self.L.dabgpu_autocfg_push_fibs(self.h, fibs.ctypes.data, fibs.shape[0], fibs.strides[0], None if ok is None else ok.ctypes.data)
        if rc < 0:
            _check(rc)
        return rc

    def dump(self) -> Tuple[np.ndarray, np.ndarray]:
        subs = np.zeros((64, 9), dtype=np.int32)
        comps = np.zeros((512, 10), dtype=np.int32)
        ns, nc = C.c_int(0), C.c_int(0)
        _check(self.L.dabgpu_autocfg_dump(self.h, subs.ctypes.data, 64, C.byref(ns), comps.ctypes.data, 512, C.byref(nc)))
        return subs[:ns.value].copy(), comps[:nc.value].copy()

    def runnable(self) -> Tuple[list, list]:
        arr = (SubchannelC * 64)()
        ids = np.zeros(64, dtype=np.uint8)
        n = C.c_int(0)
        _check(self.L.dabgpu_autocfg_runnable(self.h, arr, ids.ctypes.data, 64, C.byref(n)))
        out = [{f: getattr(arr[i], f) for f, _ in SubchannelC._fields_} for i in range(n.value)]
        return out, [int(x) for x in ids[:n.value]]

    def applied(self) -> list:
        """SubChIds that got a decoder through apply(), in sub_index order."""
        ids = np.zeros(64, dtype=np.uint8)
        n = C.c_int(0)
        _check(self.L.dabgpu_autocfg_applied(self.h, ids.ctypes.data, 64, C.byref(n)))
        return [int(x) for x in ids[:n.value]]

    def apply(self, ctx: "DabGpu", stream: int = 0) -> bool:
        rc = self.L.dabgpu_autocfg_apply(self.h, ctx.h, stream)
        if rc < 0:
            _check(rc)
        return rc == 1


IQ_FILE_MODES = ["raw_u8", "raw_s8", "raw_s16l", "raw_s16b", "raw_u16l", "raw_u16b", "raw_s32l", "raw_s32b", "raw_u32l", "raw_u32b",
                 "raw_f32l", "raw_f32b", "raw_f64l", "raw_f64b"]


def iq_convert(mode: str, raw: bytes) -> np.ndarray:
    """Raw capture bytes in one of the reference's reader modes -> complex64 samples (dabgpu_iq_convert, host only)."""
    L = load_library()
    buf = np.frombuffer(raw, dtype=np.uint8)
    out = np.empty(buf.size + 2, dtype=np.float32)
    n = C.c_size_t(0)
    _check(L.dabgpu_iq_convert(mode.encode(), buf.ctypes.data if buf.size else None, buf.size, out.ctypes.data, out.size, C.byref(n)))
    m = n.value - (n.value % 2)
    return out[:m].view(np.complex64).copy()


def softbits_to_bytes(bits: np.ndarray) -> np.ndarray:
    L = load_library()
    bits = np.ascontiguousarray(bits, dtype=np.int8)
    out = np.empty(bits.size // 8, dtype=np.uint8)
    _check(L.dabgpu_softbits_to_bytes(bits.ctypes.data, bits.size, out.ctypes.data))
    return out


def bytes_to_softbits(b: np.ndarray) -> np.ndarray:
    L = load_library()
    b = np.ascontiguousarray(b, dtype=np.uint8)
    out = np.empty(b.size * 8, dtype=np.int8)
    _check(L.dabgpu_bytes_to_softbits(b.ctypes.data, b.size, out.ctypes.data))
    return out
