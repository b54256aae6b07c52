"""Recordings, knob sets and Process() partitions shared by tests/test_ofdm_config_cpu.py (every case changes what the oracle
computes) and tests/test_ofdm_config_gpu.py (the GPU computes what the oracle computes in every case).

The synchronisation knobs of OFDM_Demod_Config (ofdm_demodulator.h:24-45, dabgpu_ofdm_config) and the partition of the input
into Process() blocks both steer the decisions of the reference's state machine.  Each recording batch mixes SNRs, carrier
frequency offsets and a noise-only stream so that every knob set below changes the oracle's output on at least one stream of
its batch (tests/test_ofdm_config_cpu.py checks that, so a GPU build that ignored a knob or the partition fails the GPU test).
"""
import importlib

import numpy as np

PKG = "sdrplusplus-dab-radio-plugin_b200"

FFT = {1: 2048, 2: 512, 3: 256, 4: 1024}
N_FRAMES = {1: 6, 2: 16, 3: 16, 4: 8}
LEAD = {1: 2000, 2: 2000, 3: 5000, 4: 2000}
SNRS = (3.0, 12.0, 20.0)
CFOS = (0.3, 2.5, 20.2)            # carrier spacings
CALL = 65536                       # samples per Process() call of the knob matrix (the CLI's block size)

# one recording per (snr, cfo) + a noise-only stream
STREAMS = [(snr, cfo) for snr in SNRS for cfo in CFOS] + [(None, 0.0)]

# knob sets: name -> (overrides, or a function of the mode for knobs given in FFT bins)
KNOBS = {
    "coarse_off": dict(is_coarse_freq_correction=0),
    "max_coarse_0": dict(max_coarse_freq_correction_norm=0.0),
    "max_coarse_4bins": lambda mode: dict(max_coarse_freq_correction_norm=4.5 / FFT[mode]),   # the 20.2-carrier stream lies beyond
    "slow_beta_1": dict(coarse_freq_slow_beta=1.0),
    "slow_beta_0.02": dict(coarse_freq_slow_beta=0.02),
    "fine_beta_0.3": dict(fine_freq_update_beta=0.3),
    "fine_beta_1": dict(fine_freq_update_beta=1.0),
    "impulse_10dB": dict(impulse_peak_threshold_db=10.0),
    "impulse_30dB": dict(impulse_peak_threshold_db=30.0),
    "distance_prob_0": dict(impulse_peak_distance_probability=0.0),
    "distance_prob_1": dict(impulse_peak_distance_probability=1.0),
    "null_0.1_0.9": dict(null_thresh_start=0.1, null_thresh_end=0.9),
    "null_0.6_0.65": dict(null_thresh_start=0.6, null_thresh_end=0.65),
    "l1_1x1": dict(signal_l1_nb_samples=1, signal_l1_nb_decimate=1),
    "l1_37x1": dict(signal_l1_nb_samples=37, signal_l1_nb_decimate=1),
    "l1_100x1": dict(signal_l1_nb_samples=100, signal_l1_nb_decimate=1),
    "l1_1000x2": dict(signal_l1_nb_samples=1000, signal_l1_nb_decimate=2),
    "l1_beta_0.5": dict(signal_l1_update_beta=0.5),
    "l1_beta_0.999": dict(signal_l1_update_beta=0.999),
}
# Each mode's knob sets apply on top of a base.  Mode III never locks on these recordings at the defaults (its fine-time peak
# stays below 20 dB): with the impulse threshold at 10 dB it does, which brings its frequency loops under test.  In mode I the
# 3 dB streams never find the NULL at the default thresholds: at 0.6 / 0.65 they do, and the impulse threshold then matters.
BASE = {1: dict(null_thresh_start=0.6, null_thresh_end=0.65), 2: {}, 3: dict(impulse_peak_threshold_db=10.0), 4: {}}
# Knob sets not run in a mode.  In modes I and IV the fine-time peak of every recording stands so far above the rest of the
# impulse response that the distance weighting never moves it: the distance knobs change nothing there (modes II and III cover
# them).  In mode III a 30 dB impulse threshold replaces the base's 10 dB and gives the defaults' output again (never locked).
# Mode III with distance probability 1 locks the 20.2-carrier streams onto wrong coarse offsets: frames are demodulated at a
# frequency word near -0.48 cycle per sample, where the PLL phase n * f of apply_pll reaches 2e4 cycles and its float32 rounding
# makes the soft bits depend on the last bit of f -- one ulp more in the oracle's own f moves 2942 soft bits of frame 4 by more
# than one step (max 23), exactly the difference the GPU shows with f within 2e-6.  A tie, not a discrepancy: not run.
EXCLUDED = {1: ("distance_prob_0", "distance_prob_1"), 3: ("impulse_30dB", "distance_prob_1"),
            4: ("distance_prob_0", "distance_prob_1")}
# c32 input runs the general L1 loop at every window length: a reduced set is enough there
KNOBS_C32 = ["coarse_off", "slow_beta_0.02", "impulse_30dB", "null_0.1_0.9", "l1_37x1", "l1_beta_0.5"]

# the non-default knob set the partition cases also run with: an odd L1 window on the u8 general loop
PARTITION_KNOBS = "l1_37x1"


def knob_cases(mode: int, c32: bool = False):
    names = KNOBS_C32 if c32 else list(KNOBS)
    return [k for k in names if k not in EXCLUDED.get(mode, ())]


def knobs(name: str, mode: int) -> dict:
    k = KNOBS[name]
    return k(mode) if callable(k) else dict(k)


def case_config(name: str, mode: int) -> dict:
    return {**BASE[mode], **knobs(name, mode)}


def params(mode: int):
    return importlib.import_module(PKG).get_params(mode)


def recordings(mode: int, n_frames: int = 0) -> np.ndarray:
    """[streams, 2 * n] u8 IQ of the batch: the same transmission impaired per stream, cut to a common length"""
    tx = importlib.import_module(PKG + ".synth.dabtx")
    sub = tx.Subchannel(0, 0, 48, eep_level=2, dabplus=False)
    ens = tx.EnsembleTx(mode, [sub], seed=500 + mode)
    base = tx.ofdm_modulate([ens.next_frame_bits() for _ in range(n_frames or N_FRAMES[mode])], mode)
    recs = []
    for i, (snr, cfo) in enumerate(STREAMS):
        if snr is None:
            rng = np.random.default_rng(900 + mode)
            x = ((rng.standard_normal(base.size + LEAD[mode] + 3000) + 1j * rng.standard_normal(base.size + LEAD[mode] + 3000))
                 * np.sqrt(0.5)).astype(np.complex64)
        else:
            x = tx.impair(base, snr, cfo / FFT[mode], LEAD[mode] + 37 * i, seed=31 * i + mode, tail_samples=3000)
        recs.append(tx.to_u8(x, 30.0))
    n = min(r.size for r in recs) // 2
    return np.stack([r[:2 * n] for r in recs])


def to_c32(u8: np.ndarray) -> np.ndarray:
    """QuantisedIQToFloatIQ<uint8_t> (app_iq_readers.h:23-43): the c32 stream the u8 path converts to on the device"""
    f = (u8.astype(np.float32) - np.float32(127.5)) * np.float32(1.0 / 127.5)
    return np.ascontiguousarray(f).view(np.complex64)


def calls(n: int, call: int = CALL):
    """[(offset, length)] of consecutive calls of `call` samples covering n samples, the last one partial"""
    return [(o, min(call, n - o)) for o in range(0, n, call)]


# Process() partitions: name -> (call lengths, block_size, limit), lengths in samples; the list of call lengths repeats until the
# input ends (limit > 0: after `limit` samples).  block_size 0 = each call is one block (the C++ adapter's OFDM_Demod::Process).
# 64 and 99 are shorter than the L1 window (UpdateSignalAverage does nothing), block size 1 only runs over a short stretch.
def partitions(mode: int) -> dict:
    P = params(mode)
    tsym, tnull, frame = P.nb_symbol_period, P.nb_null_period, P.nb_frame_samples
    return {
        "block_1": ([20000], 1, 20000),
        "block_64": ([4 * 65536], 64, 0),
        "block_99": ([4 * 65536], 99, 0),
        "block_100": ([4 * 65536], 100, 0),
        "block_101": ([4 * 65536], 101, 0),
        "block_997": ([65536], 997, 0),
        "block_tnull": ([65536], tnull, 0),
        "block_tsym": ([65536], tsym, 0),
        "block_tsym+1": ([65536], tsym + 1, 0),
        "block_frame": ([3 * frame], frame, 0),
        "block_4099": ([5 * 4099 + 17], 4099, 0),
        "block_65537": ([3 * 65537 - 5], 65537, 0),
        "ragged_calls": ([5, 99, 4099, 65536, 1, 12345, 30011], 0, 0),
        "ragged_blocks": ([70001, 12345, 99999], 997, 0),
    }


# the partitions that also run on c32 input
PARTITIONS_C32 = ["block_99", "block_997", "block_tsym+1", "ragged_calls"]
# (mode, partition, knob set) whose oracle output equals the one of the CALL-sample blocks: not run
PARTITION_NO_TEETH = {(3, "block_frame", PARTITION_KNOBS)}


def partition_cases(mode: int, c32: bool = False):
    """[(partition, knob set or None for the base)]"""
    names = PARTITIONS_C32 if c32 else list(partitions(mode))
    return [(p, k) for p in names for k in ((None,) if c32 else (None, PARTITION_KNOBS)) if (mode, p, k) not in PARTITION_NO_TEETH]


def partition_calls(n: int, lengths, limit: int = 0):
    """[(offset, length)] of the calls of a partition over n samples (limit > 0: stop after `limit` samples)"""
    out, off, i = [], 0, 0
    end = min(n, limit) if limit else n
    while off < end:
        ln = min(lengths[i % len(lengths)], end - off)
        out.append((off, ln))
        off += ln
        i += 1
    return out


def ring_for_block(mode: int, block: int) -> int:
    """the smallest power-of-two ring_samples a context accepts whose headroom (ofdm_ring_headroom: ring - frame - NULL - symbol
    - 1024) holds one block: windows and frames then straddle the ring's wrap every few frames"""
    P = params(mode)
    keep = P.nb_frame_samples + P.nb_null_period + P.nb_symbol_period
    ring = 1
    while ring < keep + 4096 or ring - keep - 1024 < block:
        ring *= 2
    return ring


def oracle_outputs(pyref, mode: int, iq: np.ndarray, cfg: dict, call_list, block_size: int, u8: bool = True,
                   use_ref: bool = False, edits=None):
    """Runs one oracle per stream over the calls; edits = {call index: knob overrides applied before that call}.
    Returns per stream {"status": [state dict after each call], "frames": [(bits, coarse, fine, time offset)]}."""
    out = []
    for s in range(iq.shape[0]):
        o = pyref.RefOfdm(mode, 1) if use_ref else pyref.PortOfdm(mode)
        if cfg:
            o.set_config(**cfg)
        st, fr = [], []
        for k, (off, ln) in enumerate(call_list):
            if edits and k in edits:
                o.set_config(**edits[k])
            chunk = iq[s, 2 * off:2 * (off + ln)] if u8 else iq[s, off:off + ln]
            pyref.ofdm_process_call(o, chunk, block_size, u8=u8)
            st.append(o.state())
            fr += o.pop_frames()
        out.append({"status": st, "frames": fr})
    return out


# Live changes (the reference's GUI edits OFDM_Demod::GetConfig() while the demodulator runs, ofdm_demodulator.h:122): calls of
# LIVE_CALL samples after a short first call that ends in the leading noise, while every stream still searches the NULL.
LIVE_CALL = 8192


def live_calls(n: int):
    return [(0, 1000)] + [(o, min(LIVE_CALL, n - o)) for o in range(1000, n, LIVE_CALL)]


# the knobs the live changes start from: BASE, except in mode IV, where a desync happens only at the end of the recordings at
# the defaults; a 30 dB impulse threshold makes some streams lose lock midway
LIVE_BASE = {**BASE, 4: dict(impulse_peak_threshold_db=30.0)}


def live_scenarios(mode: int, run) -> dict:
    """name -> {call index: knob overrides applied before that call, to every stream}, placed from the per-call states of `run`
    (the oracle over live_calls under LIVE_BASE[mode]): while the NULL is searched, in the middle of a frame, right after a desync,
    and coarse correction switched off and on again (the coarse_found / slow-beta path)."""
    st = [r["status"] for r in run]
    n_calls = len(st[0])
    ref = next(s for s in range(len(run)) if len(run[s]["frames"]) >= 2)

    def first(pred, start=1):
        return next(k for k in range(start, n_calls - 1) if pred(k))

    mid = first(lambda k: st[ref][k - 1]["state"] == 4 and st[ref][k - 1]["frames_read"] >= 1)
    desync = first(lambda k: any(x[k - 1]["frames_desync"] > x[k - 2]["frames_desync"] for x in st), start=2)
    frame_calls = -(-params(mode).nb_frame_samples // LIVE_CALL)
    return {
        "null_search": {1: dict(null_thresh_start=0.45, null_thresh_end=0.7, signal_l1_update_beta=0.9)},
        "mid_frame": {mid: dict(fine_freq_update_beta=0.3, coarse_freq_slow_beta=0.02)},
        "after_desync": {desync: dict(signal_l1_nb_samples=37, signal_l1_nb_decimate=1, impulse_peak_threshold_db=15.0)},
        "coarse_toggle": {mid: dict(is_coarse_freq_correction=0), mid + 2 * frame_calls: dict(is_coarse_freq_correction=1)},
    }


# The C++ OFDM_Demod adapter copies OFDM_Demod_Config into dabgpu_ofdm_config field by field (host/dab_adapters.hpp push_config).
# Its test edits every field between Process() calls of varying lengths; the values are all distinct, so that exchanging any two
# fields of the same type in that copy changes the oracle's output on one of the recordings (tests/test_ofdm_config_cpu.py).
ADAPTER_MODE = 2
ADAPTER_STREAMS = (1, 4)               # 3 and 12 dB at 2.5 carriers
ADAPTER_BLOCKS = [5000, 8192, 997, 30011, 65536, 12345]
ADAPTER_EDITS = {
    2: dict(signal_l1_update_beta=0.9, signal_l1_nb_samples=37, signal_l1_nb_decimate=3, null_thresh_start=0.5,
            null_thresh_end=0.7, fine_freq_update_beta=0.6, is_coarse_freq_correction=1, max_coarse_freq_correction_norm=0.004,
            coarse_freq_slow_beta=0.05, impulse_peak_threshold_db=12.0, impulse_peak_distance_probability=0.25),
    30: dict(signal_l1_update_beta=0.8, signal_l1_nb_samples=64, signal_l1_nb_decimate=2, null_thresh_start=0.55,
             null_thresh_end=0.65, fine_freq_update_beta=0.75, is_coarse_freq_correction=0, max_coarse_freq_correction_norm=0.3,
             coarse_freq_slow_beta=0.2, impulse_peak_threshold_db=14.0, impulse_peak_distance_probability=0.95),
}
FLOAT_KNOBS = ["signal_l1_update_beta", "null_thresh_start", "null_thresh_end", "fine_freq_update_beta",
               "max_coarse_freq_correction_norm", "coarse_freq_slow_beta", "impulse_peak_threshold_db",
               "impulse_peak_distance_probability"]
INT_KNOBS = ["signal_l1_nb_samples", "signal_l1_nb_decimate", "is_coarse_freq_correction"]


# tolerances of the comparison with the GPU (tests/test_ofdm_config_gpu.py)
L1_RTOL = 1e-5
FREQ_ATOL = 2e-6


def differs(a, b, per_call: bool = True) -> bool:
    """True if two oracle runs differ by more than the GPU comparison tolerates on at least one stream.  per_call: compare the
    status after every call (the runs have the same calls), else after the last one only (different partitions)."""
    for ra, rb in zip(a, b):
        if len(ra["frames"]) != len(rb["frames"]) or any(fa[3] != fb[3] for fa, fb in zip(ra["frames"], rb["frames"])):
            return True
        pairs = zip(ra["status"], rb["status"]) if per_call else [(ra["status"][-1], rb["status"][-1])]
        for sa, sb in pairs:
            if (sa["state"], sa["frames_read"], sa["frames_desync"], sa["fine_time_offset"]) != \
                    (sb["state"], sb["frames_read"], sb["frames_desync"], sb["fine_time_offset"]):
                return True
            if abs(sa["signal_avg"] - sb["signal_avg"]) > L1_RTOL * max(abs(sa["signal_avg"]), abs(sb["signal_avg"])):
                return True
            if abs(sa["coarse"] - sb["coarse"]) > FREQ_ATOL or abs(sa["fine"] - sb["fine"]) > FREQ_ATOL:
                return True
        for fa, fb in zip(ra["frames"], rb["frames"]):
            if abs(fa[1] - fb[1]) > FREQ_ATOL or abs(fa[2] - fb[2]) > FREQ_ATOL:
                return True
    return False
