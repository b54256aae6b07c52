"""Wideband front end over long runs (dabgpu_wideband_process): at five rates with different FFT pass lists and steps, and at
the smallest output capacity (2^18, passes of 66 to 154 blocks) and at 2^20 (passes of 512 blocks), enough input that the input
ring and the output ring each wrap at least twice, one call longer than twice the input ring and one that yields more outputs
than the capacity.  After every call the outputs it produced that the buffer still holds are compared with the float64
contract, evaluated on a window of the input around them (reference_outputs), so every ring wrap and pass boundary is checked."""
import numpy as np
import pytest

from test_wideband_rates_cpu import FS_OUT, MARGIN, plan, reference_outputs
from test_wideband_rates_gpu import n_out_after, open_any

pytestmark = pytest.mark.gpu

# 2.4 MS/s: 1 024 bins, steps 1 050 -> 896; 8.748: N_in 2 x 3^7, 2 187 -> 512; 12.5: 3 125 -> 512, a 50 % step; 20: 512 bins,
# 3 750 -> 384; 8.192: k_wideband<4>
LONG_RATES = [2400000, 8748000, 12500000, 20000000, 8192000]
RMS_LSB = 3000.0


def ring_geometry(dab, fs, cap):
    """dabgpu_wideband_process's bounds, restated: the OFDM headroom of the output ring, the blocks of one filter-bank pass
    and the input ring (wb_ring_log2: the history of the next block plus max_pass_blocks + 1 blocks, rounded up to a power of
    two)"""
    P = dab.get_params(1)
    p = plan(fs)
    headroom = cap - P.nb_frame_samples - P.nb_null_period - P.nb_symbol_period - 1024
    max_pass_blocks = min(512, headroom // p["step_out"])
    need = p["fft_in"] - p["step_in"] + (max_pass_blocks + 1) * p["step_in"]
    return headroom, max_pass_blocks, 1 << (need - 1).bit_length()


def call_sizes(fs, cap, ring, si):
    """a short call, one longer than twice the input ring and than the output ring, then calls of about a third of the output
    ring with a 1-sample call and a few-block call between them, until both rings wrapped at least twice"""
    per_cap = cap * fs // FS_OUT                 # input samples per output-ring length
    sizes = [12345, max(2 * ring, per_cap + per_cap // 4) + 777]
    k = 0
    while sum(sizes) <= 2 * ring or n_out_after(fs, sum(sizes)) <= 2 * cap + cap // 8:
        sizes.append([per_cap // 3 + 1, 1, 3 * si + 5][k % 3])
        k += 1
    return sizes


@pytest.mark.parametrize("cap_log2", [18, 20])
@pytest.mark.parametrize("fs", LONG_RATES)
def test_long_run_across_ring_wraps(gpu_ctx, fs, cap_log2):
    dab, fmt, cap = gpu_ctx, "raw_s16l", 1 << cap_log2
    p = plan(fs)
    si, so, d, lim = p["step_in"], p["step_out"], p["bin_hz"], fs // 2 - 768000
    headroom, max_pass_blocks, ring = ring_geometry(dab, fs, cap)
    bs = 32768 if cap_log2 == 18 else 65536      # a Process() block and a filter-bank block must fit the headroom
    assert bs + so <= headroom
    sizes = call_sizes(fs, cap, ring, si)
    n_total = sum(sizes)
    rng = np.random.default_rng(fs % 4099 + cap_log2)
    raw = np.empty((2, 2 * (n_total + MARGIN)), dtype="<i2")
    for a in range(0, raw.shape[1], 1 << 22):
        v = rng.standard_normal((2, min(1 << 22, raw.shape[1] - a))) * (RMS_LSB / np.sqrt(2))
        raw[:, a: a + v.shape[1]] = np.clip(np.round(v), -32767, 32767)
    rms_in = RMS_LSB / 32767.0

    def x_at(s):
        return lambda a, b: (raw[s, 2 * a: 2 * b: 2] + 1j * raw[s, 2 * a + 1: 2 * b: 2]) / 32767.0

    chans = [(1, -11 * d // 2), (0, -lim + 6001)]   # a rounding tie; near the band edge, off the bin grid
    g, w, out = open_any(dab, fs, fmt, [c[0] for c in chans], [c[1] for c in chans], cap=cap)
    done, n_done = 0, 0
    for n in sizes:
        got = w.process(np.ascontiguousarray(raw[:, 2 * done: 2 * (done + n)]), block_size=bs)
        done += n
        n_hi = n_out_after(fs, done)
        assert got == n_hi - n_done
        n_lo = max(n_done, n_hi - cap)           # what the buffer still holds of this call's outputs
        if n_hi > n_lo:
            o = out.cpu().numpy()
            for lo in range(n_lo, n_hi, 1 << 18):
                hi = min(n_hi, lo + (1 << 18))
                idx = np.arange(lo, hi) % cap
                for c, (s, f) in enumerate(chans):
                    err = np.abs(o[c, idx].astype(np.complex128) - reference_outputs(x_at(s), fs, f, lo, hi)) / rms_in
                    assert np.sqrt(np.mean(err ** 2)) <= 1e-4 and err.max() <= 5e-4, (done, lo, c, f, np.sqrt(np.mean(err ** 2)), err.max())
        n_done = n_hi
    # both rings wrapped at least twice, one call ran more than one pass, one yielded more than the output ring holds
    assert n_total > 2 * ring and n_done > 2 * cap
    assert max(sizes) > 2 * ring and max(sizes) // si > max_pass_blocks
    assert max(n_out_after(fs, sum(sizes[:i + 1])) - n_out_after(fs, sum(sizes[:i])) for i in range(len(sizes))) > cap
    w.close()
    g.close()
