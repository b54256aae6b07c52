"""What collecting the DAB+ access units costs on the benchmark's full-chain workload: Mode I, 1 024 streams, 18 DAB+ sub-channels
(EEP 3-A, 48 CU) each, u8 IQ from pinned host memory, one transmission frame per ticket, two tickets in flight.  One context runs
three arms, A and B alternated in rounds:
  A  dabgpu_submit with chan_status_host only (no DAB+ output);
  B  dabgpu_submit_ex with the DAB+ output of every (stream, sub-channel) copied into pinned buffers (k_dabplus_pack);
  C  the route without the batched output, over a few frames: a synchronous ticket, then dabgpu_chan_get_dabplus_events for
     every (stream, sub-channel).
Prints one JSON line per arm: median and p90 wall-clock time per ticket, AUs delivered per second (the au_ok counter delta, 0
where nothing is delivered), DAB+ bytes copied to the host per ticket, the DAB+ kernel time per call from the library's
profile counters (k_dabplus alone in A, k_dabplus + k_dabplus_pack in B, hence the pack = B - A, measured in separate profiled
tickets after the timed ones), and the GPU name and power limit read in the same run.  Needs a GPU; writes nothing."""
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
PERIOD, BLOCK = 10, 65536


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=1024)
    ap.add_argument("--tickets", type=int, default=120, help="timed tickets per arm (A and B), split over --rounds")
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=12)
    ap.add_argument("--profiled", type=int, default=20, help="profiled tickets per arm for the kernel times")
    ap.add_argument("--sync-frames", type=int, default=3, help="frames of arm C")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("dabplus_out_measure.py needs a CUDA device: the library has no CPU fallback")
    dab = importlib.import_module(PKG)
    tx = importlib.import_module(PKG + ".synth.dabtx")
    synth = importlib.import_module(PKG + ".synth.gpusynth")
    S, FS = a.streams, tx.MODES[1].nb_frame_samples
    subs = tx.default_ensemble()
    payload = np.stack([tx.periodic_frames(1, subs, seed=1000 + u, period_frames=PERIOD) for u in range(2)])
    cyc, _, _ = synth.make_cyclic_streams_u8(S, payload, mode=1, seed0=1, snr_db=15.0, device="cuda:0")
    hb = dab.HostBuffer(S * 2 * PERIOD * FS)
    h = hb.array.reshape(S, 2 * PERIOD * FS)
    torch.from_numpy(h).copy_(cyc)
    del cyc
    torch.cuda.synchronize()
    g = dab.DabGpu(mode=1, max_streams=S)
    for s in range(S):
        g.msc_configure(s, subs)
    bound = g.dabplus_out_bound(0, S)
    index_bytes = S * g.max_subchannels * 8
    status = [dab.HostBuffer(S * 8) for _ in range(2)]
    logs = [dab.HostBuffer(bound) for _ in range(2)]
    index = [dab.HostBuffer(index_bytes) for _ in range(2)]
    step = [0]

    def submit(dabplus):
        i, step[0] = step[0], step[0] + 1
        view = h[:, 2 * (i % PERIOD) * FS:2 * ((i % PERIOD) + 1) * FS]
        dp = (logs[i % 2].ptr.value, bound, index[i % 2].ptr.value) if dabplus else None
        return g.submit(view.ctypes.data, h.strides[0], FS, block_size=BLOCK, run_chan_decode=True, dabplus=dp,
                        chan_status_host=status[i % 2].ptr.value)

    def drive(n, dabplus, stamps=None):
        """n tickets, two in flight; stamps gets the time each ticket retired"""
        prev = None
        for _ in range(n):
            t = submit(dabplus)
            if prev is not None:
                g.wait(prev)
                if stamps is not None:
                    stamps.append(time.perf_counter())
            prev = t
        g.wait(prev)
        if stamps is not None:
            stamps.append(time.perf_counter())

    drive(a.warmup, False)
    drive(a.warmup, True)
    per = max(1, a.tickets // a.rounds)
    times = {"A": [], "B": []}
    aus = {"A": 0, "B": 0}
    wall = {"A": 0.0, "B": 0.0}
    for _ in range(a.rounds):
        for arm in ("A", "B"):
            c0 = g.counters()
            stamps = [time.perf_counter()]
            drive(per, arm == "B", stamps)
            times[arm] += np.diff(np.array(stamps)).tolist()
            wall[arm] += stamps[-1] - stamps[0]
            aus[arm] += g.counters()["au_ok"] - c0["au_ok"]
    prof = {}
    for arm in ("A", "B"):
        g.profile_enable(True)
        drive(a.profiled, arm == "B")
        p = g.profile_read()["dabplus"]
        g.profile_enable(False)
        prof[arm] = (p["ms"] / a.profiled, p["launches"])
    gpu = gpu_info()
    pack_ms = prof["B"][0] - prof["A"][0]
    for arm in ("A", "B"):
        t = np.array(times[arm]) * 1e3
        print(json.dumps({"arm": arm, "route": "dabgpu_submit, chan_status only" if arm == "A" else "dabgpu_submit_ex with DAB+ output",
                          "streams": S, "tickets": len(t), "ms_per_ticket_median": round(float(np.median(t)), 3),
                          "ms_per_ticket_p90": round(float(np.percentile(t, 90)), 3),
                          "aus_delivered_per_s": round(aus[arm] / wall[arm], 1) if arm == "B" else 0.0,
                          "dabplus_bytes_to_host_per_ticket": bound + index_bytes if arm == "B" else 0,
                          "dabplus_kernels_ms_per_ticket": round(prof[arm][0], 4), "dabplus_kernel_launches": prof[arm][1],
                          "k_dabplus_pack_ms_per_call": round(pack_ms, 4) if arm == "B" else None, "gpu": gpu}), flush=True)
    # arm C: synchronous ticket, then the per-sub getter for every DAB+ sub-channel of every stream
    t_c, bytes_c, au_c = [], 0, 0
    for _ in range(a.sync_frames):
        c0 = g.counters()
        t0 = time.perf_counter()
        g.wait(submit(False))
        for s in range(S):
            for k in range(len(subs)):
                log = g.get_dabplus_events(s, k)
                n_ev, has_payload, off = 0, False, 0
                while off < len(log):
                    n = int(np.frombuffer(log, dtype=np.int32, count=1, offset=off + 20)[0])
                    n_ev, has_payload, off = n_ev + 1, has_payload or n > 0, off + 24 + ((n + 3) & ~3)
                bytes_c += 4 + 32 * n_ev + (5 * dab.CIF_OUT_STRIDE if has_payload else 0)   # what the getter copies
        t_c.append(time.perf_counter() - t0)
        au_c += g.counters()["au_ok"] - c0["au_ok"]
    t = np.array(t_c) * 1e3
    print(json.dumps({"arm": "C", "route": "synchronous ticket + dabgpu_chan_get_dabplus_events per (stream, sub-channel)", "streams": S,
                      "tickets": len(t), "ms_per_ticket_median": round(float(np.median(t)), 3),
                      "ms_per_ticket_p90": round(float(np.percentile(t, 90)), 3), "aus_delivered_per_s": round(au_c / t.sum() * 1e3, 1),
                      "dabplus_bytes_to_host_per_ticket": bytes_c // max(1, len(t)), "getter_calls_per_ticket": S * len(subs),
                      "gpu": gpu}), flush=True)
    g.close()
    for b in status + logs + index + [hb]:
        b.close()


if __name__ == "__main__":
    main()
