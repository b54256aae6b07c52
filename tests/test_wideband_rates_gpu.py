"""Wideband front end at the tuners' own rates (dabgpu_wideband_open_any_rate, k_wideband_mixed) on the GPU: parity of d_out with
the float64 long-FFT evaluation of the header's contract at 2.4 to 20 MS/s in every format, bit-identical output to
dabgpu_wideband_open at 2.048 MHz x 2^d, bit-identical output however the input is split into calls, no phase drift over 2^27
input samples, round trips of synthetic multi-ensemble captures through the whole chain, and argument validation."""
import numpy as np
import pytest

from test_wideband_gpu import CAP, PERIOD, SCALE, WARM, _hash, _tx, dequantize
from test_wideband_rates_cpu import FS_OUT, plan, reference, split_offset, taps

pytestmark = pytest.mark.gpu

RATES = [2400000, 2500000, 3000000, 6000000, 10000000, 12500000, 20000000]
FORMATS = ["raw_u8", "raw_s8", "raw_s16l", "raw_f32l"]


def noise_and_tones(n, fs, rng):
    t = np.arange(n)
    x = (rng.standard_normal(n) + 1j * rng.standard_normal(n)) / np.sqrt(2)
    for f, a in ((-0.31 * fs, 0.5), (0.123 * fs, 0.7), (0.47 * fs, 0.3)):
        x = x + a * np.exp(2j * np.pi * f * t / fs)
    return x


def open_any(dab, fs, fmt, sources, offsets, cap=CAP, any_rate=True):
    import torch
    g = dab.DabGpu(mode=1, max_streams=len(sources), iq_format=dab.IQ_C32)
    out = torch.zeros((len(sources), cap), dtype=torch.complex64, device="cuda:0")
    w = g.wideband_open(fs, fmt, sources, offsets, out.data_ptr(), cap, any_rate=any_rate)
    return g, w, out


def n_out_after(fs, n_in):
    p = plan(fs)
    return p["step_out"] * (n_in // p["step_in"])


@pytest.mark.parametrize("fs", RATES)
@pytest.mark.parametrize("fmt", FORMATS)
def test_parity_with_formula(gpu_ctx, fs, fmt):
    import torch
    p = plan(fs)
    rng = np.random.default_rng(fs % 7919 + FORMATS.index(fmt))
    n_in = p["step_in"] * 40 + 1234
    n_tot = n_in + 20000                      # the reference's interpolation near the last output sees realistic input after it
    raws, xs = [], []
    for _ in range(2):
        raw = _tx().quantize(noise_and_tones(n_tot, fs, rng), fmt, 0.25 if fmt == "raw_f32l" else SCALE[fmt] / 5)
        raws.append(raw)
        xs.append(dequantize(raw, fmt))
    lim = fs // 2 - 768000
    d = p["bin_hz"]
    sources = [0, 0, 0, 1, 1, 1]
    offsets = [-lim, d // 2 - 1 - 2 * d, lim - d // 2, -lim + d + 777, 6001, lim]
    g, w, out = open_any(gpu_ctx, fs, fmt, sources, offsets)
    got_n = w.process(np.stack(raws), block_size=65536)
    assert got_n == n_out_after(fs, n_tot)
    n_out = n_out_after(fs, n_in)
    torch.cuda.synchronize()
    got = out[:, :n_out].cpu().numpy().astype(np.complex128)
    for c, (s, f) in enumerate(zip(sources, offsets)):
        ref = reference(xs[s], fs, f)[:n_out]
        rms_in = np.sqrt(np.mean(np.abs(xs[s]) ** 2))
        err = np.abs(got[c] - ref) / rms_in
        assert np.sqrt(np.mean(err ** 2)) <= 1e-4 and err.max() <= 5e-4, (c, f, np.sqrt(np.mean(err ** 2)), err.max())
    w.close()
    g.close()


@pytest.mark.parametrize("D", [1, 4, 16])
def test_same_output_as_power_of_two_entry_point(gpu_ctx, D):
    import torch
    fs, fmt = D * FS_OUT, "raw_s16l"
    rng = np.random.default_rng(50 + D)
    n_in = 448 * D * 30 + 999
    raw = np.stack([_tx().quantize(noise_and_tones(n_in, fs, rng), fmt, 3000.0) for _ in range(2)])
    lim = fs // 2 - 768000
    sources, offsets = [0, 0, 1, 1], [-lim, 1999 - 4000 * D, 6001, lim]
    g1, w1, out1 = open_any(gpu_ctx, fs, fmt, sources, offsets, any_rate=False)
    g2, w2, out2 = open_any(gpu_ctx, fs, fmt, sources, offsets)
    n1, n2 = w1.process(raw), w2.process(raw)
    assert n1 == n2 == 448 * (n_in // (448 * D))
    torch.cuda.synchronize()
    assert torch.equal(out1[:, :n1].view(torch.float32), out2[:, :n2].view(torch.float32))
    for o in (w1, g1, w2, g2):
        o.close()


@pytest.mark.parametrize("fs", [10000000, 2400000])
def test_call_partition_invariance(gpu_ctx, fs):
    import torch
    fmt = "raw_s16l"
    rng = np.random.default_rng(fs % 101)
    n_in = 600000
    raw = np.stack([_tx().quantize(noise_and_tones(n_in, fs, rng), fmt, 3000.0) for _ in range(2)])
    lim = fs // 2 - 768000
    sources, offsets = [0, 1, 1], [-lim + 1234, 0, lim - 4321]
    g1, w1, out1 = open_any(gpu_ctx, fs, fmt, sources, offsets)
    assert w1.process(raw) == n_out_after(fs, n_in)
    g2, w2, out2 = open_any(gpu_ctx, fs, fmt, sources, offsets)
    done, total = 0, 0
    for n in (1, 4095, 65536, 333333, n_in - 1 - 4095 - 65536 - 333333):
        got = w2.process(np.ascontiguousarray(raw[:, 2 * done: 2 * (done + n)]))
        assert got == n_out_after(fs, done + n) - n_out_after(fs, done)
        done += n
        total += got
    assert total == n_out_after(fs, n_in)
    torch.cuda.synchronize()
    assert torch.equal(out1[:, :total].view(torch.float32), out2[:, :total].view(torch.float32))
    for o in (w1, g1, w2, g2):
        o.close()


def test_no_phase_drift(gpu_ctx):
    import torch
    fs = 10000000
    f_k = 1712000 + 1234                       # 1234 Hz off the 2 kHz grid of this rate
    f_tone = f_k + 5000
    g, w, out = open_any(gpu_ctx, fs, "raw_f32l", [0], [f_k])
    chunk = 1 << 22
    n_total = 1 << 27
    for k in range(n_total // chunk):
        m = np.arange(k * chunk, (k + 1) * chunk, dtype=np.int64)
        x = np.exp(2j * np.pi * ((f_tone * m) % fs) / fs) * 0.5
        raw = np.empty((1, 2 * chunk), dtype="<f4")
        raw[0, 0::2], raw[0, 1::2] = x.real, x.imag
        w.process(raw, block_size=65536)
    n_out = n_out_after(fs, n_total)
    torch.cuda.synchronize()
    n = np.arange(n_out - 4096, n_out, dtype=np.int64)
    got = out[0, torch.from_numpy(n % CAP).to(out.device)].cpu().numpy().astype(np.complex128)
    h = taps(fs)
    _, delta = split_offset(f_k, plan(fs)["bin_hz"])
    Hd = np.sum(h * np.exp(-2j * np.pi * (delta + 5000) * np.arange(h.size) / fs))
    want = 0.5 * Hd * np.exp(2j * np.pi * ((5000 * n) % FS_OUT) / FS_OUT)
    dphi = np.angle(got * np.conj(want))
    assert np.abs(dphi).max() < 1e-3, np.abs(dphi).max()
    assert np.abs(np.abs(got) / np.abs(want) - 1).max() < 1e-3
    w.close()
    g.close()


# ---- round trips through the whole chain ----------------------------------------------------------------------------------
def make_capture(tx, fs, offsets, seeds, gains_db=(), seed=0):
    subs = tx.default_ensemble()[:4]
    made = [tx.periodic_frames(1, subs, seed=sd, period_frames=PERIOD, return_logical=True) for sd in seeds]
    rng = np.random.default_rng(seed)
    cfo = [float(v) for v in rng.uniform(-8000, 8000, len(offsets))]
    shifts = [int(v) for v in rng.integers(0, PERIOD * tx.MODES[1].nb_frame_samples, len(offsets))]
    cap = tx.wideband_capture(1, [m[0] for m in made], 1, offsets, snr_db=15.0, cfo_hz=cfo, shifts=shifts, gains_db=gains_db,
                              seed=seed, sample_rate=fs)
    return cap, [m[1] for m in made]


def round_trip(dab, tx, fs, fmt, rms, captures, source_map, channels, seed):
    """as test_wideband_gpu.round_trip, at any rate: one frame's worth of input per call (0.096 fs samples), every frame
    channel-decoded; over the last PERIOD + 1 calls every channel must give back the transmitted logical frames of every
    sub-channel in transmission order, each once per period, with every FIB CRC good and no RS, fire-code or AU-CRC failure."""
    import torch
    subs = tx.default_ensemble()[:4]
    FS = tx.MODES[1].nb_frame_samples
    raws = [tx.quantize(cap, fmt, rms).reshape(-1, 2) for cap, _ in captures]
    n_ch = len(channels)
    g = dab.DabGpu(mode=1, max_streams=n_ch, iq_format=dab.IQ_C32)
    cap_out = 1 << 19
    out = torch.zeros((n_ch, cap_out), dtype=torch.complex64, device="cuda:0")
    w = g.wideband_open(fs, fmt, [c[0] for c in channels], [c[1] for c in channels], out.data_ptr(), cap_out,
                        n_sources=len(source_map), any_rate=True)
    for c in range(n_ch):
        g.msc_configure(c, subs)
    rng = np.random.default_rng(seed)
    wts = rng.integers(1, 2 ** 63, size=256, dtype=np.uint64) | np.uint64(1)
    got = [[[] for _ in subs] for _ in range(n_ch)]
    c_start = None
    step = FS * fs // FS_OUT
    for i in range(WARM + PERIOD + 1):
        block = np.stack([np.take(raws[ci], np.arange(lead + i * step, lead + (i + 1) * step), axis=0, mode="wrap").reshape(-1)
                          for ci, lead in source_map])
        n_out = w.process(block, block_size=65536)
        assert n_out == n_out_after(fs, (i + 1) * step) - n_out_after(fs, i * step)
        if i == WARM:
            c_start = g.counters()
        while True:
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


BAND3_10M = [-3424000, -1712000, 0, 1712000, 3424000]


def test_round_trip_rtl_2_4_u8_off_centre(gpu_ctx, tx):
    cap = make_capture(tx, 2400000, [-200000], [51], seed=11)
    round_trip(gpu_ctx, tx, 2400000, "raw_u8", 30.0, [cap], [(0, 0)], [(0, -200000, 0)], seed=11)


def test_round_trip_6m_s8_three_ensembles(gpu_ctx, tx):
    offs = [-1712000, 0, 1712000]
    cap = make_capture(tx, 6000000, offs, [52, 53, 54], seed=12)
    round_trip(gpu_ctx, tx, 6000000, "raw_s8", 40.0, [cap], [(0, 0)], [(0, f, e) for e, f in enumerate(offs)], seed=12)


def test_round_trip_10m_s16_five_ensembles_one_weak(gpu_ctx, tx):
    cap = make_capture(tx, 10000000, BAND3_10M, [61 + k for k in range(5)], gains_db=[0, 0, 0, -20, 0], seed=13)
    round_trip(gpu_ctx, tx, 10000000, "raw_s16l", 3000.0, [cap], [(0, 0)], [(0, f, e) for e, f in enumerate(BAND3_10M)], seed=13)


def test_round_trip_12_5m_f32_half_step_plan(gpu_ctx, tx):
    p = plan(12500000)
    assert 2 * p["step_out"] == p["fft_out"]
    offs = [-3424000, 0, 5136000]
    cap = make_capture(tx, 12500000, offs, [71, 72, 73], seed=14)
    round_trip(gpu_ctx, tx, 12500000, "raw_f32l", 0.25, [cap], [(0, 0)], [(0, f, e) for e, f in enumerate(offs)], seed=14)


def test_round_trip_32_sources_10m_five_ensembles(gpu_ctx, tx):
    caps = [make_capture(tx, 10000000, BAND3_10M, [81 + 5 * u + k for k in range(5)], seed=15 + u) for u in range(2)]
    step = tx.MODES[1].nb_frame_samples * 10000000 // FS_OUT
    source_map = [(s % 2, (s * 7919 * 37) % (PERIOD * step)) for s in range(32)]
    channels = [(s, f, e) for s in range(32) for e, f in enumerate(BAND3_10M)]
    round_trip(gpu_ctx, tx, 10000000, "raw_s16l", 3000.0, caps, source_map, channels, seed=15)


# ---- validation ----------------------------------------------------------------------------------------------------------
BAD_RATES = (2047000, 2100000, 7000000, 9375000, 32769000, 0, -10000000)


def test_errors(gpu_ctx):
    import torch
    dab = gpu_ctx
    out = torch.zeros((4, CAP), dtype=torch.complex64, device="cuda:0")

    def rc_of(g, rate=10000000, offsets=(1712000, -1712000), cap=CAP):
        try:
            w = g.wideband_open(rate, "raw_s16l", [0, 0], list(offsets), out.data_ptr(), cap, any_rate=True)
        except dab.DabGpuError as e:
            return e.code, str(e)
        w.close()
        return dab.OK, ""

    g = dab.DabGpu(mode=1, max_streams=4, iq_format=dab.IQ_C32)
    for rate in BAD_RATES:
        assert rc_of(g, rate=rate)[0] == dab.ERR_INVALID, rate
        with pytest.raises(dab.DabGpuError):
            dab.wideband_plan(rate)
    for rate in (2400000, 3000000, 10000000, 20000000):
        lim = rate // 2 - 768000
        assert rc_of(g, rate=rate, offsets=(lim + 1, 0))[0] == dab.ERR_INVALID
        assert rc_of(g, rate=rate, offsets=(0, -lim - 1))[0] == dab.ERR_INVALID
        assert rc_of(g, rate=rate, offsets=(lim, -lim))[0] == dab.OK
    P = dab.get_params(1)
    for rate in (2500000, 10000000, 20000000):
        min_cap = P.nb_frame_samples + P.nb_null_period + P.nb_symbol_period + 1024 + plan(rate)["step_out"]
        rc, msg = rc_of(g, rate=rate, offsets=(0, 0), cap=1 << 17)
        assert rc == dab.ERR_INVALID and f"[{min_cap}, 2^30]" in msg, msg
        assert rc_of(g, rate=rate, offsets=(0, 0), cap=1 << 18)[0] == dab.OK
        assert rc_of(g, rate=rate, offsets=(0, 0), cap=(1 << 18) + 1)[0] == dab.ERR_INVALID
    w = g.wideband_open(10000000, "raw_s16l", [0, 0], [0, 0], out.data_ptr(), CAP, any_rate=True)
    assert rc_of(g)[0] == dab.ERR_STATE
    w.close()
    g.close()
    g_u8 = dab.DabGpu(mode=1, max_streams=4)
    assert rc_of(g_u8)[0] == dab.ERR_INVALID
    g_u8.close()
