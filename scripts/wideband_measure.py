"""Wideband front end at full size: 128 sources x 16.384 MS/s x 8 ensembles (+-0.856, +-2.568, +-4.280, +-5.992 MHz) = 1 024 Mode I
streams, one transmission frame (96 ms of signal) per step.  Prints one JSON line per input format with the step time of
process + chan_decode (CUDA events), the channelizer kernel time from torch.profiler in a separate run, the achieved FLOP/s and
bytes/s of the kernel, and the host->device rate.  Needs a GPU; writes nothing but the traces asked for with --out."""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PKG = "sdrplusplus-dab-radio-plugin_b200"
OFFS = [-5992000, -4280000, -2568000, -856000, 856000, 2568000, 4280000, 5992000]
D, S, PERIOD = 8, 128, 5


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def design_counts(n_in, bps):
    """FLOP and bytes per step by design arithmetic: 5 N log2 N per complex FFT, 6 per complex multiply."""
    N = 512 * D
    blocks = n_in // (448 * D)
    fwd = 5 * N * np.log2(N)
    per_chan = 5 * 512 * 9 + 512 * 12 + 448 * 6
    flop = S * blocks * (fwd + len(OFFS) * per_chan)
    byts = S * blocks * (N * bps + len(OFFS) * 448 * 8)
    return float(flop), float(byts)


def run(fmt, steps, warmup, out_dir):
    import torch
    dab = importlib.import_module(PKG)
    tx = importlib.import_module(PKG + ".synth.dabtx")
    bps = dab.WB_BYTES_PER_SAMPLE[dab.WB_FORMATS[fmt]]
    FS = tx.MODES[1].nb_frame_samples
    subs = tx.default_ensemble()
    made = [tx.periodic_frames(1, subs, seed=900 + k, period_frames=PERIOD) for k in range(2)]
    cap = tx.wideband_capture(1, [made[k % 2] for k in range(8)], D, OFFS, snr_db=15.0, cfo_hz=[1500.0 * (k - 4) for k in range(8)],
                              shifts=[37117 * k for k in range(8)], seed=5)
    raw = tx.quantize(cap, fmt, 3000.0 if fmt == "raw_s16l" else 28.0).view(np.uint8).reshape(-1, bps)
    step = D * FS
    # every source holds PERIOD + 1 frames of the periodic capture from its own lead, so step i reads frame i mod PERIOD
    hb = dab.HostBuffer(S * (PERIOD + 1) * step * bps)
    h = hb.array.reshape(S, (PERIOD + 1) * step * bps)
    for s in range(S):
        idx = (np.arange((PERIOD + 1) * step) + 104729 * s) % raw.shape[0]
        h[s] = raw[idx].reshape(-1)
    g = dab.DabGpu(mode=1, max_streams=S * len(OFFS), iq_format=dab.IQ_C32)
    out = torch.zeros((S * len(OFFS), 1 << 19), dtype=torch.complex64, device="cuda:0")
    w = g.wideband_open(D * 2048000, fmt, [s for s in range(S) for _ in OFFS], OFFS * S, out.data_ptr(), 1 << 19)
    for c in range(S * len(OFFS)):
        g.msc_configure(c, subs)

    def one(i):
        v = h[:, (i % PERIOD) * step * bps: ((i % PERIOD) + 1) * step * bps]
        w.process(v, block_size=65536)
        g.chan_decode()

    for i in range(warmup):
        one(i)
    g.sync()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    stream = torch.cuda.ExternalStream(g.cuda_stream)
    ms = []
    for i in range(warmup, warmup + steps):
        g.chan_join()
        ev[0].record(stream)
        one(i)
        g.chan_join()
        ev[1].record(stream)
        ev[1].synchronize()
        ms.append(ev[0].elapsed_time(ev[1]))
    c = g.counters()
    # H2D alone: the same bytes as one step, pinned
    d_tmp = torch.empty(S * step * bps, dtype=torch.uint8, device="cuda:0")
    src = torch.from_numpy(h[:, :step * bps].reshape(-1))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(5):
        d_tmp.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    h2d_gbs = 5 * S * step * bps / (time.perf_counter() - t0) / 1e9
    del d_tmp
    # kernel time from the profiler, separate run
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(warmup + steps, warmup + steps + 10):
            one(i)
        g.sync()
    k_us = [e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total for e in prof.key_averages() if "k_wideband" in e.key]
    k_n = [e.count for e in prof.key_averages() if "k_wideband" in e.key]
    if out_dir:
        prof.export_chrome_trace(os.path.join(out_dir, f"wideband_trace_{fmt}.json"))
    kernel_ms = sum(k_us) / 1000.0 / 10
    flop, byts = design_counts(step, bps)
    res = dict(metric="wideband_front_end", gpu=gpu_info(), format=fmt, sources=S, streams=S * len(OFFS), sample_rate=D * 2048000,
               step_signal_ms=FS / 2048.0, steps=steps, step_ms_median=float(np.median(ms)), step_ms_p90=float(np.percentile(ms, 90)),
               channelizer_kernel_ms_per_step=kernel_ms, channelizer_launches_per_step=sum(k_n) / 10,
               kernel_tflops=flop / (kernel_ms * 1e-3) / 1e12, kernel_tbytes_s=byts / (kernel_ms * 1e-3) / 1e12,
               design_gflop_per_step=flop / 1e9, design_gbytes_per_step=byts / 1e9, h2d_gbytes_s=h2d_gbs,
               h2d_ms_per_step=S * step * bps / h2d_gbs / 1e6, realtime_streams=S * len(OFFS) * (FS / 2048.0) / float(np.median(ms)),
               frames_demodulated=c["frames_demodulated"], fibs_crc_ok=c["fibs_crc_ok"], fibs_total=c["fibs_total"],
               superframes_rs_fail=c["superframes_rs_fail"], au_crc_fail=c["au_crc_fail"])
    w.close()
    g.close()
    hb.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--formats", default="raw_s16l,raw_s8")
    ap.add_argument("--out", default=None, help="directory for the profiler's chrome traces (none written if omitted)")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("wideband_measure.py needs a CUDA device")
    if a.out:
        os.makedirs(a.out, exist_ok=True)
    for fmt in a.formats.split(","):
        print(json.dumps(run(fmt, a.steps, a.warmup, a.out)), flush=True)


if __name__ == "__main__":
    main()
