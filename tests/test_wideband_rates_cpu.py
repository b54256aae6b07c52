"""Wideband front end at any tuner rate (dabgpu_wideband_plan, dabgpu_wideband_open_any_rate), CPU side: the library's plan
agrees with a restatement of the rule in include/dabgpu.h at every multiple of 1 kHz, the channel filter meets its mask at every
supported rate, and a numpy model of the mixed-radix filter bank the kernel implements (k_wideband_mixed, wideband.cuh) agrees
with a float64 long-FFT evaluation of the header's output contract."""
from math import ceil, gcd, log2

import numpy as np
import pytest
from scipy import signal

FS_OUT = 2048000


def plan(fs):
    """the header's rule: of the bin spacings 4, 2, 1 kHz that divide fs with fs / bin <= 8192 and 5-smooth, the fewest
    inverse-FFT operations per output sample; None where no spacing qualifies"""
    if fs < FS_OUT or fs > 16 * FS_OUT:
        return None
    best = None
    for d in (4000, 2000, 1000):
        if fs % d:
            continue
        n_in, m = fs // d, fs // d
        for p in (2, 3, 5):
            while m % p == 0:
                m //= p
        if n_in > 8192 or m != 1:
            continue
        n_out = FS_OUT // d
        T = 2 * ceil(fs / 64000) + 1
        ov_out = -(-(T - 1) * FS_OUT // fs)
        g = FS_OUT // gcd(fs, FS_OUT)
        lcm = g * 64 // gcd(g, 64)
        step_out = (n_out - ov_out) // lcm * lcm
        if step_out <= 0:
            continue
        cost = 5 * n_out * log2(n_out) / step_out
        if best is None or cost < best[0]:
            best = (cost, dict(bin_hz=d, fft_in=n_in, fft_out=n_out, step_in=step_out * fs // FS_OUT, step_out=step_out, taps=T))
    return None if best is None else best[1]


GRID = [f for f in range(FS_OUT, 16 * FS_OUT + 1, 1000)]
SUPPORTED = [f for f in GRID if plan(f)]
MODEL_RATES = [2400000, 2500000, 3000000, 6000000, 10000000, 12500000, 20000000, 2250000, 8000000]


def taps(fs):
    return signal.firwin(plan(fs)["taps"], 856e3, window=("kaiser", signal.kaiser_beta(70)), fs=fs)


def split_offset(f, d):
    """f = d b + delta, b rounded half away from zero"""
    b = (f + d // 2) // d if f >= 0 else -((d // 2 - f) // d)
    return b, f - d * b


def reference(x, fs, f):
    """the header's contract in float64 over one long FFT: mix by f^, filter with the DFT of h, keep |f| < 1.024 MHz, evaluate
    at input times n fs / 2.048 MHz, rotate by delta.  x holds input beyond the outputs asked for, so the tail is realistic."""
    p = plan(fs)
    b, delta = split_offset(f, p["bin_hz"])
    m = np.arange(x.size, dtype=np.int64)
    z = x * np.exp(-2j * np.pi * ((b * m) % p["fft_in"]) / p["fft_in"])
    q = fs // gcd(fs, FS_OUT)                        # P a multiple of q: P * 2.048 MHz / fs is an integer
    P = -(-(x.size + p["taps"]) // q) * q
    Q = P * FS_OUT // fs
    V = np.fft.fft(z, P) * np.fft.fft(taps(fs), P)
    k = np.fft.fftfreq(P, 1.0 / P).astype(np.int64)
    keep = np.abs(k) * fs < FS_OUT // 2 * P
    Y = np.zeros(Q, dtype=np.complex128)
    Y[k[keep] % Q] = V[keep]
    y = np.fft.ifft(Y) * (Q / P)
    n = np.arange(Q, dtype=np.int64)
    return y * np.exp(-2j * np.pi * ((n % FS_OUT) * delta % FS_OUT) / FS_OUT)


def model(x, fs, f):
    """the kernel's algorithm: fft_in-point FFT per block, fft_out bins around the channel (wrapping modulo fft_in) times
    H / fft_in and the block's mixing phase, fft_out-point inverse FFT, the last step_out outputs kept, rotated by delta"""
    p = plan(fs)
    N, NO, si, so = p["fft_in"], p["fft_out"], p["step_in"], p["step_out"]
    b_k, delta = split_offset(f, p["bin_hz"])
    H = np.fft.fft(taps(fs), N)
    u = np.arange(-NO // 2, NO // 2)
    nblk = x.size // si
    ov = N - si
    xp = np.concatenate([np.zeros(ov, x.dtype), x])
    out = np.empty(so * nblk, dtype=np.complex128)
    for b in range(nblk):
        a0 = b * si - ov
        S = np.fft.fft(xp[b * si: b * si + N])
        Z = np.zeros(NO, dtype=np.complex128)
        Z[u % NO] = S[(b_k + u) % N] * H[u % N] / N * np.exp(-2j * np.pi * ((b_k * a0) % N) / N)
        out[so * b: so * (b + 1)] = (np.fft.ifft(Z) * NO)[NO - so:]
    n = np.arange(out.size, dtype=np.int64)
    return out * np.exp(-2j * np.pi * ((n % FS_OUT) * delta % FS_OUT) / FS_OUT)


def test_plan_matches_library_on_every_khz(dab):
    assert len(GRID) == 30721 and len(SUPPORTED) == 105
    for fs in GRID:
        want = plan(fs)
        if want is None:
            with pytest.raises(dab.DabGpuError) as e:
                dab.wideband_plan(fs)
            assert e.value.code == dab.ERR_INVALID
        else:
            assert dab.wideband_plan(fs) == want, fs
    for fs in (2048001, 2400100, 10000500, 12345678, 20000040, 32767999, 0, -2048000, 2047000, 32769000):
        with pytest.raises(dab.DabGpuError):
            dab.wideband_plan(fs)


def test_plan_examples():
    table = {2400000: (2000, 1200, 1024, 1050, 896, 77), 2500000: (1000, 2500, 2048, 1875, 1536, 81),
             3000000: (1000, 3000, 2048, 2625, 1792, 95), 6000000: (2000, 3000, 1024, 2625, 896, 189),
             8000000: (4000, 2000, 512, 1750, 448, 251), 10000000: (2000, 5000, 1024, 4375, 896, 315),
             12500000: (2000, 6250, 1024, 3125, 512, 393), 20000000: (4000, 5000, 512, 3750, 384, 627)}
    for fs, t in table.items():
        assert tuple(plan(fs).values()) == t, fs
    for D in (1, 2, 4, 8, 16):   # the power-of-two rates keep dabgpu_wideband_open's geometry
        assert plan(D * FS_OUT) == dict(bin_hz=4000, fft_in=512 * D, fft_out=512, step_in=448 * D, step_out=448, taps=64 * D + 1)
    for fs in (2100000, 7000000, 9375000, 2047000):
        assert plan(fs) is None


def test_filter_mask_every_supported_rate():
    worst_944 = -1e9
    for fs in SUPPORTED:
        h = taps(fs)
        assert abs(h.sum() - 1.0) < 1e-12
        n = 1 << 20                                  # fs / 2^20 <= 31.25 Hz grid
        resp = np.fft.rfft(h, n)
        f = np.arange(resp.size) * fs / n
        db = 20 * np.log10(np.maximum(np.abs(resp), 1e-300))
        assert np.max(np.abs(db[f <= 768e3])) <= 0.003, fs
        worst_944 = max(worst_944, np.max(db[f >= 944e3]))
        # 944 kHz is the nearest carrier of the next block; the worst rate on this grid is 2.25 MHz at -71.15 dB
        assert np.max(db[f >= 944e3]) <= -71.1, fs
        assert np.max(db[f >= 1024e3]) <= -75.0, fs
    assert worst_944 > -71.2


@pytest.mark.parametrize("fs", MODEL_RATES)
def test_mixed_radix_model_matches_long_fft_reference(fs):
    p = plan(fs)
    rng = np.random.default_rng(fs % 9973)
    n_in = p["step_in"] * 10 + 333
    x = (rng.standard_normal(n_in + 20000) + 1j * rng.standard_normal(n_in + 20000)) / np.sqrt(2)
    lim = fs // 2 - 768000
    for f in (-lim, lim, 0, p["bin_hz"] // 2 - 1 - 2 * p["bin_hz"], 123457 % lim, -lim + 777):
        got = model(x[:n_in], fs, f)
        assert got.size == p["step_out"] * (n_in // p["step_in"])
        ref = reference(x, fs, f)[:got.size]
        err = np.abs(got - ref)
        assert np.sqrt(np.mean(err ** 2)) < 1e-5 and err.max() < 1e-4, (f, np.sqrt(np.mean(err ** 2)), err.max())


def test_model_is_the_power_of_two_formula():
    """at 2.048 MHz x D every output time is an input sample: the model is the existing overlap-save filter bank"""
    fs = 4 * FS_OUT
    rng = np.random.default_rng(4)
    n_in = 448 * 4 * 6 + 77
    x = (rng.standard_normal(n_in) + 1j * rng.standard_normal(n_in)) / np.sqrt(2)
    b, delta = split_offset(1001234, 4000)
    m = np.arange(n_in, dtype=np.int64)
    v = signal.fftconvolve(x * np.exp(-2j * np.pi * ((4000 * b * m) % fs) / fs), taps(fs))[:n_in]
    n = np.arange(448 * (n_in // (448 * 4)), dtype=np.int64)
    direct = v[:n.size * 4:4] * np.exp(-2j * np.pi * ((n * 4 % fs) * delta % fs) / fs)
    assert np.max(np.abs(model(x, fs, 1001234) - direct)) < 2e-4
