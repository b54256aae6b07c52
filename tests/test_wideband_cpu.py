"""Wideband front end (dabgpu_wideband_*), CPU side: the channel filter meets its mask at every rate, and a numpy model of the
overlap-save filter bank the kernel implements (wideband.cuh) agrees with the direct formula of the header."""
import numpy as np
import pytest
from scipy import signal

RATES = [1, 2, 4, 8, 16]


def taps(D):
    return signal.firwin(64 * D + 1, 856e3, window=("kaiser", signal.kaiser_beta(70)), fs=D * 2048000)


def split_offset(f):
    """f = 4000 b + delta, b rounded half away from zero"""
    b = (f + 2000) // 4000 if f >= 0 else -((2000 - f) // 4000)
    return b, f - 4000 * b


def direct(x, D, f):
    """y[n] = exp(-j2pi delta nD/fs) sum_i h[i] x[nD-i] exp(-j2pi f^ (nD-i)/fs), float64, phases from exact integers"""
    fs = D * 2048000
    b, delta = split_offset(f)
    m = np.arange(x.size, dtype=np.int64)
    z = x * np.exp(-2j * np.pi * ((4000 * b * m) % fs) / fs)
    v = signal.fftconvolve(z, taps(D))[:x.size]
    n_out = 448 * (x.size // (448 * D))
    n = np.arange(n_out, dtype=np.int64)
    return v[:n_out * D:D] * np.exp(-2j * np.pi * ((n * D % fs) * delta % fs) / fs)


def overlap_save(x, D, f):
    """the kernel's algorithm: N = 512 D point FFT per block, 512 bins around the channel times H, 512-point inverse FFT"""
    fs, N = D * 2048000, 512 * D
    b_k, delta = split_offset(f)
    H = np.fft.fft(taps(D), N)
    u = np.arange(-256, 256)
    nblk = x.size // (448 * D)
    xp = np.concatenate([np.zeros(64 * D, x.dtype), x])
    out = np.empty(448 * nblk, dtype=np.complex128)
    for b in range(nblk):
        S = np.fft.fft(xp[448 * D * b: 448 * D * b + N])
        Z = np.zeros(512, dtype=np.complex128)
        Z[u % 512] = S[(b_k + u) % N] * H[u % N] * np.exp(-2j * np.pi * ((b_k * (7 * b - 1)) % 8) / 8)
        out[448 * b: 448 * (b + 1)] = (np.fft.ifft(Z) * 512 / N)[64:]
    n = np.arange(out.size, dtype=np.int64)
    return out * np.exp(-2j * np.pi * ((n * D % fs) * delta % fs) / fs)


@pytest.mark.parametrize("D", RATES)
def test_filter_mask(D):
    fs = D * 2048000
    h = taps(D)
    assert h.size == 64 * D + 1 and abs(h.sum() - 1.0) < 1e-12
    f = np.linspace(0, fs / 2, 1 << 16)
    _, resp = signal.freqz(h, worN=f, fs=fs)
    db = 20 * np.log10(np.maximum(np.abs(resp), 1e-300))
    assert np.max(np.abs(db[f <= 768e3])) <= 0.003
    # 944 kHz is the nearest carrier of the next block; on this dense grid the worst rate (D = 2) reaches -71.48 dB there
    assert np.max(db[f >= 944e3]) <= -71.4
    assert np.max(db[f >= 1024e3]) <= -75.0


@pytest.mark.parametrize("D", RATES)
def test_overlap_save_model_matches_direct_formula(D):
    rng = np.random.default_rng(D)
    n_in = 448 * D * 12 + 333
    x = (rng.standard_normal(n_in) + 1j * rng.standard_normal(n_in)) / np.sqrt(2)
    lim = D * 1024000 - 768000
    for f in (-lim, 1999 - 4000 * D, lim - 2000, 123457 % (lim + 1)):
        ref, got = direct(x, D, f), overlap_save(x, D, f)
        assert got.size == ref.size == 448 * (n_in // (448 * D))
        err = np.abs(got - ref)
        if D == 1:
            assert err.max() < 1e-12
        else:
            assert np.sqrt(np.mean(err ** 2)) < 5e-5 and err.max() < 2e-4, (f, np.sqrt(np.mean(err ** 2)), err.max())


def test_offset_split_rounds_half_away_from_zero():
    assert split_offset(2000) == (1, -2000) and split_offset(-2000) == (-1, 2000)
    assert split_offset(1999) == (0, 1999) and split_offset(-6001) == (-2, 1999) and split_offset(856000) == (214, 0)
