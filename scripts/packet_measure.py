"""What two packet-mode sub-channels per stream cost on the benchmark's full-chain workload: Mode I, 1 024 streams, 18 sub-channels
(EEP 3-A, 48 CU) each, u8 IQ from pinned host memory, one transmission frame per ticket, two tickets in flight, every ticket with
the batched sub-channel output (dabgpu_submit_ex).  Two contexts on the same GPU, fed the same IQ, alternated in rounds:
  A  all 18 entries DAB+ (entries 16 and 17 carry packets, so their DAB+ stage finds no superframe there);
  B  16 DAB+ entries + 2 DABGPU_PAYLOAD_PACKET_FEC entries (k_packet, k_packet_pack);
  C  16 DAB+ entries + 2 DABGPU_PAYLOAD_PACKET entries on the same bytes: the walk, CRC and log writes of k_packet without the
     FEC ring and the RS(204,188) decode of closed sets, so k_packet's time in B minus C is what the FEC part costs.
Prints one JSON line per arm: median and p90 wall-clock time per ticket, packets delivered per second (crc_ok PACKET records of the
copied logs), the log + index bytes copied per ticket (the bound dabgpu_dabplus_out_bound sizes the copy, not what the logs hold),
the DABGPU_PROF_DABPLUS class time per ticket (k_dabplus + k_dabplus_pack, plus k_packet + k_packet_pack in B) from separately
profiled tickets, the launch count per ticket, the time of each kernel of that class per ticket from a torch.profiler pass of
its own, and the GPU name and power limit read in the same run.  periodic_frames repeats the payload every PERIOD frames: an FEC
set that crosses the seam is abandoned or fails its rows, so only the crc_ok packets are counted.  Needs a GPU; writes nothing."""
import argparse
import dataclasses
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
EV_PACKET = 6
ARMS = ("A", "B", "C")
TABLES = {"A": "18 DAB+", "B": "16 DAB+ + 2 PACKET_FEC", "C": "16 DAB+ + 2 PACKET"}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def packets_ok(dab, log, index, max_subs, keys):
    n = 0
    for key, rec in dab.split_dabplus(log, index, 0, max_subs).items():
        if key[1] not in keys:
            continue
        off = 0
        while off < len(rec):
            t, _, crc_ok, _, _, nb = np.frombuffer(rec, dtype=np.int32, count=6, offset=off)
            n += int(t == EV_PACKET and crc_ok == 1)
            off += 24 + ((int(nb) + 3) & ~3)
    return n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=1024)
    ap.add_argument("--tickets", type=int, default=120, help="timed tickets per arm, split over --rounds")
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=12)
    ap.add_argument("--profiled", type=int, default=20, help="profiled tickets per arm for the kernel class times")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("packet_measure.py needs a CUDA device: the library has no CPU fallback")
    dab = importlib.import_module(PKG)
    tx = importlib.import_module(PKG + ".synth.dabtx")
    synth = importlib.import_module(PKG + ".synth.gpusynth")
    S, FS = a.streams, tx.MODES[1].nb_frame_samples
    subs_a = tx.default_ensemble()
    subs_b = [dataclasses.replace(sc, packet_fec=True) if sc.id >= 16 else sc for sc in subs_a]
    subs_c = [dataclasses.replace(sc, packet_fec=False) if sc.id >= 16 else sc for sc in subs_a]
    payload = np.stack([tx.periodic_frames(1, subs_b, seed=1000 + u, period_frames=PERIOD) for u in range(2)])
    cyc, _, _ = synth.make_cyclic_streams_u8(S, payload, mode=1, seed0=1, snr_db=15.0, device="cuda:0")
    hb = dab.HostBuffer(S * 2 * PERIOD * FS)
    h = hb.array.reshape(S, 2 * PERIOD * FS)
    torch.from_numpy(h).copy_(cyc)
    del cyc
    torch.cuda.synchronize()
    arms = {}
    for arm, subs in (("A", subs_a), ("B", subs_b), ("C", subs_c)):
        g = dab.DabGpu(mode=1, max_streams=S)
        for s in range(S):
            g.msc_configure(s, subs)
        bound = g.dabplus_out_bound(0, S)
        arms[arm] = dict(g=g, bound=bound, step=0, logs=[dab.HostBuffer(bound) for _ in range(2)],
                         index=[dab.HostBuffer(S * g.max_subchannels * 8) for _ in range(2)], status=[dab.HostBuffer(S * 8) for _ in range(2)])

    def drive(arm, n, stamps=None, count=None):
        X = arms[arm]
        g, prev = X["g"], None

        def retire(t, j):
            g.wait(t)
            if stamps is not None:
                stamps.append(time.perf_counter())
            if count is not None:
                count[0] += packets_ok(dab, X["logs"][j].array, X["index"][j].array, g.max_subchannels, (16, 17))

        for _ in range(n):
            i = X["step"]
            X["step"] += 1
            view = h[:, 2 * (i % PERIOD) * FS:2 * ((i % PERIOD) + 1) * FS]
            t = g.submit(view.ctypes.data, h.strides[0], FS, block_size=BLOCK, run_chan_decode=True,
                         dabplus=(X["logs"][i % 2].ptr.value, X["bound"], X["index"][i % 2].ptr.value), chan_status_host=X["status"][i % 2].ptr.value)
            if prev is not None:
                retire(*prev)
            prev = (t, i % 2)
        retire(*prev)

    for arm in ARMS:
        drive(arm, a.warmup)
    per = max(1, a.tickets // a.rounds)
    times = {arm: [] for arm in ARMS}
    wall = {arm: 0.0 for arm in ARMS}
    pkts = {arm: [0] for arm in ARMS}
    for _ in range(a.rounds):
        for arm in ARMS:
            stamps = [time.perf_counter()]
            drive(arm, per, stamps)
            times[arm] += np.diff(np.array(stamps)).tolist()
            wall[arm] += stamps[-1] - stamps[0]
    for arm in ("B", "C"):
        drive(arm, per, None, pkts[arm])   # packets delivered, counted outside the timed window
    prof = {}
    for arm in ARMS:
        g = arms[arm]["g"]
        l0 = g.launch_count
        g.profile_enable(True)
        drive(arm, a.profiled)
        p = g.profile_read()["dabplus"]
        g.profile_enable(False)
        prof[arm] = (p["ms"] / a.profiled, (g.launch_count - l0) / a.profiled)
    kernels = {}
    for arm in ARMS:
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as tp:
            drive(arm, a.profiled)
        kernels[arm] = {}
        for ev in tp.key_averages():
            name = ev.key.split("(")[0].split("<")[0].replace("void ", "").strip()
            if name in ("k_dabplus", "k_dabplus_pack", "k_packet", "k_packet_pack"):
                t_us = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
                kernels[arm][name] = round(t_us / 1e3 / a.profiled, 4)
    gpu = gpu_info()
    for arm in ARMS:
        t = np.array(times[arm]) * 1e3
        X = arms[arm]
        print(json.dumps({"arm": arm, "table": TABLES[arm], "streams": S, "tickets": len(t),
                          "ms_per_ticket_median": round(float(np.median(t)), 3), "ms_per_ticket_p90": round(float(np.percentile(t, 90)), 3),
                          "packets_delivered_per_s": round(pkts[arm][0] / (per * float(np.median(t)) * 1e-3), 1) if arm != "A" else 0.0,
                          "log_bound_bytes_to_host_per_ticket": X["bound"] + S * X["g"].max_subchannels * 8,
                          "dabplus_class_ms_per_ticket": round(prof[arm][0], 4), "launches_per_ticket": prof[arm][1],
                          "kernel_ms_per_ticket": kernels[arm], "gpu": gpu}), flush=True)
    for X in arms.values():
        X["g"].close()
        for b in X["logs"] + X["index"] + X["status"]:
            b.close()
    hb.close()


if __name__ == "__main__":
    main()
