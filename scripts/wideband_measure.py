"""Wideband front end at full size: 128 sources x 16.384 MS/s x 8 ensembles (+-0.856, +-2.568, +-4.280, +-5.992 MHz) = 1 024 Mode I
streams, one transmission frame (96 ms of signal) per step.  With --rate, captures at that rate (any rate dabgpu_wideband_plan
supports, through dabgpu_wideband_open_any_rate) with the Band III offsets (multiples of 1.712 MHz) that fit it and enough
sources for about 1 024 streams, e.g. 204 sources x 5 ensembles at 10 MS/s.  Prints one JSON line per input format with the
step time of process + chan_decode (CUDA events), the channelizer kernel time from torch.profiler in a separate run, the
achieved FLOP/s and bytes/s of the kernel, the host->device rate and the rate's plan.  With --pipelined the same run also drives
the workload through dabgpu_wideband_reserve + dabgpu_wideband_submit / dabgpu_wait on a second context, two tickets in flight,
each with its channel decode and the channel status and MSC bytes copied into pinned buffers, as a receiver would, and adds the
wall-clock time per ticket, the real-time streams it gives, the pinned host->device time of a step and whether the counter
deltas over the timed tickets equal those of the timed serial steps.  Needs a GPU; writes nothing but the traces asked for with
--out."""
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
DEFAULT_RATE = D * 2048000
STREAMS = 1024


def workload(rate):
    """(offsets, sources) of the workload at `rate`"""
    if rate == DEFAULT_RATE:
        return OFFS, S
    k = (rate // 2 - 768000) // 1712000
    offs = [1712000 * j for j in range(-k, k + 1)]
    return offs, STREAMS // len(offs)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def design_counts(n_in, bps, plan, offs, n_src):
    """FLOP and bytes per step by design arithmetic: 5 N log2 N per complex FFT, 6 per complex multiply; every block reads its
    fft_in input samples and writes step_out c32 outputs per channel."""
    N, NO, so = plan["fft_in"], plan["fft_out"], plan["step_out"]
    blocks = n_in // plan["step_in"]
    fwd = 5 * N * np.log2(N)
    per_chan = 5 * NO * np.log2(NO) + NO * 12 + so * 6
    flop = n_src * blocks * (fwd + len(offs) * per_chan)
    byts = n_src * blocks * (N * bps + len(offs) * so * 8)
    return float(flop), float(byts)


COUNTERS = ("frames_demodulated", "fibs_crc_ok", "fibs_total", "superframes_ok", "superframes_rs_fail", "au_ok", "au_crc_fail")


def delta(c1, c0):
    return {k: c1[k] - c0[k] for k in COUNTERS}


def run_pipelined(dab, h, hb, S, E, offs, subs, fmt, rate, step, bps, steps, warmup, out_dir):
    """the serial leg's steps as tickets of dabgpu_wideband_submit on a fresh context: (wall-clock ms per ticket, counter deltas
    over the timed tickets)"""
    import torch
    g = dab.DabGpu(mode=1, max_streams=S * E, iq_format=dab.IQ_C32)
    out = torch.zeros((S * E, 1 << 19), dtype=torch.complex64, device="cuda:0")
    w = g.wideband_open(rate, fmt, [s for s in range(S) for _ in offs], offs * S, out.data_ptr(), 1 << 19,
                        any_rate=rate != DEFAULT_RATE)
    for c in range(S * E):
        g.msc_configure(c, subs)
    w.reserve(step)
    nc = g.P.nb_cifs
    outs = [(dab.HostBuffer(S * E * 8), dab.HostBuffer(S * E * nc * dab.CIF_OUT_STRIDE)) for _ in range(2)]
    row = h.strides[0]

    def submit(i):
        st, msc = outs[i % 2]
        return w.submit(hb.ptr.value + (i % PERIOD) * step * bps, row, step, block_size=65536, run_chan_decode=True,
                        chan_status_host=st.ptr.value, msc_host=msc.ptr.value)

    def drive(first, n, stamps=None):
        prev = None
        for i in range(first, first + n):
            t = submit(i)
            if prev is not None:
                g.wait(prev)
                if stamps is not None:
                    stamps.append(time.perf_counter())
            prev = t
        g.wait(prev)
        if stamps is not None:
            stamps.append(time.perf_counter())

    drive(0, warmup)
    c0 = g.counters()
    stamps = [time.perf_counter()]
    drive(warmup, steps, stamps)
    c1 = g.counters()
    if out_dir:
        from torch.profiler import profile, ProfilerActivity
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            drive(warmup + steps, 10)
        name = f"wideband_pipelined_trace_{fmt}.json" if rate == DEFAULT_RATE else f"wideband_pipelined_trace_{rate}_{fmt}.json"
        prof.export_chrome_trace(os.path.join(out_dir, name))
    w.close()
    g.close()
    for a, b in outs:
        a.close()
        b.close()
    return np.diff(np.array(stamps)) * 1e3, delta(c1, c0)


def run(fmt, steps, warmup, out_dir, rate=DEFAULT_RATE, pipelined=False):
    import torch
    dab = importlib.import_module(PKG)
    tx = importlib.import_module(PKG + ".synth.dabtx")
    bps = dab.WB_BYTES_PER_SAMPLE[dab.WB_FORMATS[fmt]]
    FS = tx.MODES[1].nb_frame_samples
    subs = tx.default_ensemble()
    plan = dab.wideband_plan(rate)
    offs, S = workload(rate)
    E = len(offs)
    made = [tx.periodic_frames(1, subs, seed=900 + k, period_frames=PERIOD) for k in range(2)]
    if rate == DEFAULT_RATE:
        cap = tx.wideband_capture(1, [made[k % 2] for k in range(8)], D, OFFS, snr_db=15.0, cfo_hz=[1500.0 * (k - 4) for k in range(8)],
                                  shifts=[37117 * k for k in range(8)], seed=5)
    else:
        cap = tx.wideband_capture(1, [made[k % 2] for k in range(E)], 1, offs, snr_db=15.0,
                                  cfo_hz=[1500.0 * (k - E // 2) for k in range(E)], shifts=[37117 * k for k in range(E)], seed=5,
                                  sample_rate=rate)
    raw = tx.quantize(cap, fmt, 3000.0 if fmt == "raw_s16l" else 28.0).view(np.uint8).reshape(-1, bps)
    step = FS * rate // 2048000
    # every source holds PERIOD + 1 frames of the periodic capture from its own lead, so step i reads frame i mod PERIOD
    hb = dab.HostBuffer(S * (PERIOD + 1) * step * bps)
    h = hb.array.reshape(S, (PERIOD + 1) * step * bps)
    for s in range(S):
        idx = (np.arange((PERIOD + 1) * step) + 104729 * s) % raw.shape[0]
        h[s] = raw[idx].reshape(-1)
    g = dab.DabGpu(mode=1, max_streams=S * E, iq_format=dab.IQ_C32)
    out = torch.zeros((S * E, 1 << 19), dtype=torch.complex64, device="cuda:0")
    w = g.wideband_open(rate, fmt, [s for s in range(S) for _ in offs], offs * S, out.data_ptr(), 1 << 19,
                        any_rate=rate != DEFAULT_RATE)
    for c in range(S * E):
        g.msc_configure(c, subs)

    def one(i):
        v = h[:, (i % PERIOD) * step * bps: ((i % PERIOD) + 1) * step * bps]
        w.process(v, block_size=65536)
        g.chan_decode()

    for i in range(warmup):
        one(i)
    g.sync()
    c_timed = g.counters()
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
    serial_delta = delta(c, c_timed)
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
        name = f"wideband_trace_{fmt}.json" if rate == DEFAULT_RATE else f"wideband_trace_{rate}_{fmt}.json"
        prof.export_chrome_trace(os.path.join(out_dir, name))
    kernel_ms = sum(k_us) / 1000.0 / 10
    flop, byts = design_counts(step, bps, plan, offs, S)
    res = dict(metric="wideband_front_end", gpu=gpu_info(), format=fmt, sources=S, streams=S * E, sample_rate=rate, plan=plan,
               step_signal_ms=FS / 2048.0, steps=steps, step_ms_median=float(np.median(ms)), step_ms_p90=float(np.percentile(ms, 90)),
               channelizer_kernel_ms_per_step=kernel_ms, channelizer_launches_per_step=sum(k_n) / 10,
               kernel_tflops=flop / (kernel_ms * 1e-3) / 1e12, kernel_tbytes_s=byts / (kernel_ms * 1e-3) / 1e12,
               design_gflop_per_step=flop / 1e9, design_gbytes_per_step=byts / 1e9, h2d_gbytes_s=h2d_gbs,
               h2d_ms_per_step=S * step * bps / h2d_gbs / 1e6, realtime_streams=S * E * (FS / 2048.0) / float(np.median(ms)),
               frames_demodulated=c["frames_demodulated"], fibs_crc_ok=c["fibs_crc_ok"], fibs_total=c["fibs_total"],
               superframes_rs_fail=c["superframes_rs_fail"], au_crc_fail=c["au_crc_fail"])
    w.close()
    g.close()
    if pipelined:
        # the same step's bytes from the pinned buffer (the line above copies a pageable copy of them)
        d_tmp = torch.empty(S * step * bps, dtype=torch.uint8, device="cuda:0")
        src = torch.from_numpy(hb.array[:S * step * bps])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(5):
            d_tmp.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        pinned_h2d_ms = (time.perf_counter() - t0) / 5 * 1e3
        del d_tmp
        pms, pipe_delta = run_pipelined(dab, h, hb, S, E, offs, subs, fmt, rate, step, bps, steps, warmup, out_dir)
        res.update(pipelined_tickets=steps, pipelined_step_ms_median=float(np.median(pms)), pipelined_step_ms_p90=float(np.percentile(pms, 90)),
                   pipelined_step_ms_mean=float(np.mean(pms)), pipelined_realtime_streams=S * E * (FS / 2048.0) / float(np.median(pms)),
                   pinned_h2d_ms_per_step=pinned_h2d_ms, serial_counter_deltas=serial_delta, pipelined_counter_deltas=pipe_delta,
                   pipelined_counters_equal=pipe_delta == serial_delta)
    hb.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--formats", default="raw_s16l,raw_s8")
    ap.add_argument("--rate", type=int, default=DEFAULT_RATE, help="capture rate in Hz (default: 16.384 MHz, 128 x 8 ensembles)")
    ap.add_argument("--out", default=None, help="directory for the profiler's chrome traces (none written if omitted)")
    ap.add_argument("--pipelined", action="store_true", help="also time the workload through reserve + submit / wait (two tickets in flight)")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("wideband_measure.py needs a CUDA device")
    if a.out:
        os.makedirs(a.out, exist_ok=True)
    for fmt in a.formats.split(","):
        print(json.dumps(run(fmt, a.steps, a.warmup, a.out, a.rate, a.pipelined)), flush=True)


if __name__ == "__main__":
    main()
