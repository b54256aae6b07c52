"""Wideband front end (dabgpu_wideband_*) on the GPU: parity of d_out with the float64 formula of the header at every rate and
format, bit-identical output however the input is split into calls, no phase drift over 2^27 input samples, round trips of
synthetic multi-ensemble captures through the whole chain, and argument validation."""
import importlib

import numpy as np
import pytest
from scipy import signal

pytestmark = pytest.mark.gpu

RATES = [1, 2, 4, 8, 16]
FORMATS = ["raw_u8", "raw_s8", "raw_s16l", "raw_f32l"]
SCALE = {"raw_u8": 127.5, "raw_s8": 127.0, "raw_s16l": 32767.0}
CAP = 1 << 19   # leaves the OFDM stage room for Process() blocks of 65 536 samples


def taps(D):
    return signal.firwin(64 * D + 1, 856e3, window=("kaiser", signal.kaiser_beta(70)), fs=D * 2048000)


def split_offset(f):
    b = (f + 2000) // 4000 if f >= 0 else -((2000 - f) // 4000)
    return b, f - 4000 * b


def direct(x, D, f):
    """the header's formula in float64, phases from exact integers"""
    fs = D * 2048000
    b, delta = split_offset(f)
    m = np.arange(x.size, dtype=np.int64)
    v = signal.fftconvolve(x * np.exp(-2j * np.pi * ((4000 * b * m) % fs) / fs), taps(D))[:x.size]
    n = np.arange(448 * (x.size // (448 * D)), dtype=np.int64)
    return v[:n.size * D:D] * np.exp(-2j * np.pi * ((n * D % fs) * delta % fs) / fs)


def dequantize(raw, fmt):
    """what the library reads: dabgpu_iq_convert's scaling"""
    v = raw.astype(np.float64)
    if fmt == "raw_u8":
        v = (v - 127.5) / 127.5
    elif fmt != "raw_f32l":
        v = v / SCALE[fmt]
    return v[0::2] + 1j * v[1::2]


def noise_and_tones(n, D, rng):
    fs = D * 2048000
    t = np.arange(n)
    x = (rng.standard_normal(n) + 1j * rng.standard_normal(n)) / np.sqrt(2)
    for f, a in ((-0.31 * fs, 0.5), (0.123 * fs, 0.7), (0.47 * fs, 0.3)):
        x = x + a * np.exp(2j * np.pi * f * t / fs)
    return x


def open_front_end(dab, D, fmt, sources, offsets, n_ch=None, cap=CAP, mode=1):
    import torch
    g = dab.DabGpu(mode=mode, max_streams=n_ch or len(sources), iq_format=dab.IQ_C32)
    out = torch.zeros((len(sources), cap), dtype=torch.complex64, device="cuda:0")
    w = g.wideband_open(D * 2048000, fmt, sources, offsets, out.data_ptr(), cap)
    return g, w, out


@pytest.mark.parametrize("D", RATES)
@pytest.mark.parametrize("fmt", FORMATS)
def test_parity_with_formula(gpu_ctx, D, fmt):
    import torch
    rng = np.random.default_rng(100 * D + FORMATS.index(fmt))
    lim = D * 1024000 - 768000
    n_in = 448 * D * 40 + 1234
    raws, xs = [], []
    for s in range(2):
        x = noise_and_tones(n_in, D, rng)
        raw = _tx().quantize(x, fmt, 0.25 if fmt == "raw_f32l" else SCALE[fmt] / 5)
        raws.append(raw)
        xs.append(dequantize(raw, fmt))
    sources = [0, 0, 0, 1, 1, 1]
    offsets = [-lim, 1999 - 4000 * D, lim - 2000, -lim + 4000 + 777, 6001, lim]
    g, w, out = open_front_end(gpu_ctx, D, fmt, sources, offsets)
    n_out = w.process(np.stack(raws), block_size=65536)
    assert n_out == 448 * (n_in // (448 * D))
    torch.cuda.synchronize()
    got = out[:, :n_out].cpu().numpy().astype(np.complex128)
    for c, (s, f) in enumerate(zip(sources, offsets)):
        ref = direct(xs[s], D, f)
        rms_in = np.sqrt(np.mean(np.abs(xs[s]) ** 2))
        err = np.abs(got[c] - ref) / rms_in
        assert np.sqrt(np.mean(err ** 2)) <= 1e-4 and err.max() <= 5e-4, (c, f, np.sqrt(np.mean(err ** 2)), err.max())
    w.close()
    g.close()


def _tx():
    return importlib.import_module("sdrplusplus-dab-radio-plugin_b200.synth.dabtx")


def test_call_partition_invariance(gpu_ctx):
    import torch
    D, fmt = 4, "raw_s16l"
    rng = np.random.default_rng(7)
    n_in = 600000
    raw = np.stack([_tx().quantize(noise_and_tones(n_in, D, rng), fmt, 3000.0) for _ in range(2)])
    sources, offsets = [0, 1, 1], [-1712000 + 1234, 0, 1712000 - 4321]
    g1, w1, out1 = open_front_end(gpu_ctx, D, fmt, sources, offsets)
    assert w1.process(raw) == 448 * (n_in // (448 * D))
    g2, w2, out2 = open_front_end(gpu_ctx, D, fmt, sources, offsets)
    done, total = 0, 0
    for n in (1, 4095, 65536, 333333, n_in - 1 - 4095 - 65536 - 333333):
        got = w2.process(np.ascontiguousarray(raw[:, 2 * done: 2 * (done + n)]))
        assert got == 448 * ((done + n) // (448 * D)) - 448 * (done // (448 * D))
        done += n
        total += got
    assert total == 448 * (n_in // (448 * D))
    torch.cuda.synchronize()
    assert torch.equal(out1[:, :total].view(torch.float32), out2[:, :total].view(torch.float32))
    for o in (w1, g1, w2, g2):
        o.close()


def test_no_phase_drift(gpu_ctx):
    import torch
    D, fs = 8, 8 * 2048000
    f_k = 2568000 + 1234
    f_tone = f_k + 5000
    g, w, out = open_front_end(gpu_ctx, D, "raw_f32l", [0], [f_k])
    chunk = 1 << 22
    n_total = 1 << 27
    for k in range(n_total // chunk):
        m = np.arange(k * chunk, (k + 1) * chunk, dtype=np.int64)
        x = np.exp(2j * np.pi * ((f_tone * m) % fs) / fs) * 0.5
        raw = np.empty((1, 2 * chunk), dtype="<f4")
        raw[0, 0::2], raw[0, 1::2] = x.real, x.imag
        w.process(raw, block_size=65536)
    n_out = 448 * (n_total // (448 * D))
    torch.cuda.synchronize()
    n = np.arange(n_out - 4096, n_out, dtype=np.int64)
    got = out[0, torch.from_numpy(n % CAP).to(out.device)].cpu().numpy().astype(np.complex128)
    h = taps(D)
    b, delta = split_offset(f_k)
    Hd = np.sum(h * np.exp(-2j * np.pi * (delta + 5000) * np.arange(h.size) / fs))
    want = 0.5 * Hd * np.exp(2j * np.pi * ((5000 * n * D) % fs) / fs)
    dphi = np.angle(got * np.conj(want))
    assert np.abs(dphi).max() < 1e-3, np.abs(dphi).max()
    w.close()
    g.close()


# ---- round trips through the whole chain ----------------------------------------------------------------------------------
PERIOD, WARM = 5, 10


def _hash(rows, wts):
    return (rows.astype(np.uint64) * wts[None, :rows.shape[-1]]).sum(axis=-1, dtype=np.uint64)


def round_trip(dab, tx, D, fmt, rms, captures, source_map, channels, seed):
    """captures: list of (capture period complex128, logical frames per ensemble); source_map[s] = (capture, lead);
    channels[c] = (source, offset_hz, ensemble index in that capture).  Feeds one frame's worth of input per call (a call yields
    438 or 439 blocks, so a stream completes 0, 1 or 2 frames in it) and channel-decodes every frame produced.  Over the last
    PERIOD + 1 calls every channel must give back the transmitted logical frames of every sub-channel in transmission order, each
    once per period, with every FIB CRC good."""
    import torch
    subs = tx.default_ensemble()[:4]
    FS = tx.MODES[1].nb_frame_samples
    raws = [tx.quantize(cap, fmt, rms).reshape(-1, 2) for cap, _ in captures]
    n_ch = len(channels)
    g = dab.DabGpu(mode=1, max_streams=n_ch, iq_format=dab.IQ_C32)
    cap_out = 1 << 19
    out = torch.zeros((n_ch, cap_out), dtype=torch.complex64, device="cuda:0")
    w = g.wideband_open(D * 2048000, fmt, [c[0] for c in channels], [c[1] for c in channels], out.data_ptr(), cap_out,
                        n_sources=len(source_map))
    for c in range(n_ch):
        g.msc_configure(c, subs)
    rng = np.random.default_rng(seed)
    wts = rng.integers(1, 2 ** 63, size=256, dtype=np.uint64) | np.uint64(1)
    got = [[[] for _ in subs] for _ in range(n_ch)]
    c_start = None
    step = D * FS
    for i in range(WARM + PERIOD + 1):
        block = np.stack([np.take(raws[ci], np.arange(lead + i * step, lead + (i + 1) * step), axis=0, mode="wrap").reshape(-1)
                          for ci, lead in source_map])
        n_out = w.process(block, block_size=65536)
        assert n_out == 448 * (((i + 1) * step) // (448 * D)) - 448 * ((i * step) // (448 * D))
        if i == WARM:
            c_start = g.counters()
        while True:   # drain: chan_decode takes the oldest undecoded frame of every stream
            g.chan_decode()
            decoded = [c for c in range(n_ch) if g.chan_status(c)[0] == 1]
            if not decoded:
                break
            if i < WARM:
                continue
            for c in decoded:
                _, ok = g.get_fic(c)
                assert ok.all(), f"call {i}: channel {c}: a FIB failed its CRC"
                for k in range(len(subs)):
                    msc, valid = g.get_msc(c, k)
                    assert valid.all(), f"call {i}: channel {c} sub-channel {k}: a CIF is not valid"
                    got[c][k].extend(_hash(msc, wts).tolist())
    c_end = g.counters()
    d = {k: c_end[k] - c_start[k] for k in c_end}
    for c, (s, _, e) in enumerate(channels):
        logical = captures[source_map[s][0]][1][e]
        for k, sc in enumerate(subs):
            want = _hash(logical[sc.id], wts)
            seq = np.array(got[c][k], dtype=np.uint64)
            assert seq.size >= want.size, f"channel {c} sub-channel {k}: {seq.size} CIFs decoded in the window"
            j = np.nonzero(want == seq[0])[0]
            assert j.size == 1, f"channel {c} sub-channel {k}: decoded a logical frame that was not transmitted"
            assert np.array_equal(seq, want[(j[0] + np.arange(seq.size)) % want.size]), \
                f"channel {c} sub-channel {k}: decoded frames are not the transmitted ones in order, once per period"
    assert d["superframes_rs_fail"] == 0 and d["superframes_firecode_fail"] == 0 and d["au_crc_fail"] == 0
    assert d["fibs_crc_ok"] == d["fibs_total"] > 0 and d["frames_dropped"] == 0 and d["au_ok"] > 0
    w.close()
    g.close()


def make_capture(tx, D, offsets, seeds, gains_db=(), seed=0):
    subs = tx.default_ensemble()[:4]
    made = [tx.periodic_frames(1, subs, seed=sd, period_frames=PERIOD, return_logical=True) for sd in seeds]
    rng = np.random.default_rng(seed)
    cfo = [float(v) for v in rng.uniform(-8000, 8000, len(offsets))]
    shifts = [int(v) for v in rng.integers(0, PERIOD * tx.MODES[1].nb_frame_samples, len(offsets))]
    cap = tx.wideband_capture(1, [m[0] for m in made], D, offsets, snr_db=15.0, cfo_hz=cfo, shifts=shifts, gains_db=gains_db, seed=seed)
    return cap, [m[1] for m in made]


def test_round_trip_4_ensembles_s16(gpu_ctx, tx):
    offs = [-2568000, -856000, 856000, 2568000]
    cap = make_capture(tx, 4, offs, [11, 12, 13, 14], seed=1)
    round_trip(gpu_ctx, tx, 4, "raw_s16l", 3000.0, [cap], [(0, 0)], [(0, f, e) for e, f in enumerate(offs)], seed=1)


def test_round_trip_8_ensembles_s8_one_weak(gpu_ctx, tx):
    offs = [-5992000, -4280000, -2568000, -856000, 856000, 2568000, 4280000, 5992000]
    cap = make_capture(tx, 8, offs, [21 + k for k in range(8)], gains_db=[0, 0, 0, 0, -20, 0, 0, 0], seed=2)
    round_trip(gpu_ctx, tx, 8, "raw_s8", 40.0, [cap], [(0, 0)], [(0, f, e) for e, f in enumerate(offs)], seed=2)


def test_round_trip_rtl_style_u8_off_centre(gpu_ctx, tx):
    cap = make_capture(tx, 1, [-200000], [31], seed=3)
    round_trip(gpu_ctx, tx, 1, "raw_u8", 30.0, [cap], [(0, 0)], [(0, -200000, 0)], seed=3)


def test_round_trip_128_streams_32_sources(gpu_ctx, tx):
    offs = [-2568000, -856000, 856000, 2568000]
    caps = [make_capture(tx, 4, offs, [41 + 4 * u + k for k in range(4)], seed=4 + u) for u in range(2)]
    FS = tx.MODES[1].nb_frame_samples
    source_map = [(s % 2, (s * 7919 * 37) % (PERIOD * FS * 4)) for s in range(32)]
    channels = [(s, f, e) for s in range(32) for e, f in enumerate(offs)]
    round_trip(gpu_ctx, tx, 4, "raw_s16l", 3000.0, caps, source_map, channels, seed=4)


# ---- validation ----------------------------------------------------------------------------------------------------------
def test_errors(gpu_ctx):
    import torch
    dab = gpu_ctx
    out = torch.zeros((4, CAP), dtype=torch.complex64, device="cuda:0")

    def rc_of(g, rate=8192000, fmt="raw_s16l", sources=(0, 0), offsets=(856000, -856000), cap=CAP, n_sources=None):
        try:
            w = g.wideband_open(rate, fmt, list(sources), list(offsets), out.data_ptr(), cap, n_sources=n_sources)
        except dab.DabGpuError as e:
            return e.code
        w.close()
        return dab.OK

    g_u8 = dab.DabGpu(mode=1, max_streams=4)
    assert rc_of(g_u8) == dab.ERR_INVALID
    g_u8.close()
    g = dab.DabGpu(mode=1, max_streams=4, iq_format=dab.IQ_C32)
    for rate in (6144000, 10000000, 2048000 * 32, 0):
        assert rc_of(g, rate=rate) == dab.ERR_INVALID
    lim = 4096000 - 768000
    assert rc_of(g, offsets=(lim + 1, 0)) == dab.ERR_INVALID
    assert rc_of(g, offsets=(0, -lim - 1)) == dab.ERR_INVALID
    assert rc_of(g, sources=[0] * 5, offsets=[0] * 5) == dab.ERR_INVALID
    assert rc_of(g, sources=(0, 2), n_sources=2) == dab.ERR_INVALID
    assert rc_of(g, sources=(0, -1), n_sources=2) == dab.ERR_INVALID
    assert rc_of(g, cap=CAP - 1) == dab.ERR_INVALID
    assert rc_of(g, cap=1 << 17) == dab.ERR_INVALID
    assert rc_of(g, cap=1 << 18) == dab.OK
    w = g.wideband_open(8192000, "raw_s16l", [0, 0], [lim, -lim], out.data_ptr(), CAP)   # the edges themselves are valid
    assert rc_of(g) == dab.ERR_STATE
    with pytest.raises(dab.DabGpuError) as e:
        g.ofdm_process(np.zeros((1, 1024), dtype=np.complex64))
    assert e.value.code == dab.ERR_STATE
    w.close()
    assert rc_of(g) == dab.OK
    g.close()
