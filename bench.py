#!/usr/bin/env python
"""bench.py -- DAB Mode I receive-path throughput on B200 (driver contract: one JSON line on rank 0).

  python bench.py --gpus N --steps K --warmup W [--workload full|ofdm] [--streams S]
  python bench.py --impl reference ...      # the reference's own CPU implementation on the host cores
  python bench.py ... --dump-outputs DIR    # also writes what the last timed step computed to DIR/<name>.npy

Workload (BASELINE.json configs[3], the north-star target): the FULL chain -- OFDM demodulation (PRS sync, FFT, DQPSK,
frequency de-interleave) -> FIC + 18 x EEP 3-A DAB+ sub-channels (time de-interleave, de-puncture, K=7 Viterbi, energy
dispersal) -> RS(120,110) superframes -- batched over 1024 Mode I streams per GPU.  One step = every stream advances by one
transmission frame (196608 IQ samples, three Process() blocks of 65536), i.e. 201 M samples per GPU per step.

  value          device-resident throughput (inputs in HBM), CUDA events on the launching stream, max over ranks
  e2e            the same through dabgpu_submit/dabgpu_wait with pinned HOST buffers: H2D of the step's u8 IQ and D2H of the
                 decoded FIC/MSC bytes inside the timed region (>= 100 steps)
  roofline       dominant kernel of the step (by CUDA-event time of a profiled pass): algorithmic bytes / kernel time against
                 the measured HBM peak, plus issue-side figures for the Viterbi kernel (ACS/s, ALU-pipe utilisation)
  ofdm_only      the OFDM stage alone on the same streams (BASELINE configs[1]) with the roofline of k_ofdm_demod2
  spot_check     the reference chain (oracle/_ref) run on a few of the very streams the GPU decoded, outside the timed region:
                 frame / FIB / byte / superframe / access-unit counters must be identical
  cpu_baseline   the reference's CPU chain on all host cores, bounded sample (N = 1 only)

Inputs are synthetic: per stream a seeded periodic transmission (period 10 frames = 8 DAB+ superframes, valid fire codes, RS
parity and AU CRCs), its own CFO (+-20 kHz), timing lead and AWGN at 15 dB, quantised to u8 like the reference's readers do.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = "sdrplusplus-dab-radio-plugin_b200"
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FRAME_SAMPLES = 196608
BLOCK = 65536
PERIOD_FRAMES = 10                          # 40 CIFs = 8 superframes: the synthetic transmission repeats after this many frames
# SURVEY.md 8(d), per Mode I frame
OFDM_ALG_BYTES = 393216 + 230400            # u8 IQ in + int8 soft bits out
OFDM_ALG_BYTES_C32 = 1572864 + 230400       # complex<float> IQ in + int8 soft bits out (SURVEY.md section 8(d): 9.172 B/sample)
OFDM_ALG_FLOP = 17.7e6                      # floating-point operations per Mode I frame (SURVEY.md section 8(d))
VIT_ALG_BYTES = 230400 + (110592 + 3072) // 8   # soft bits in + decoded bytes out (decisions stay on chip)
VIT_STEPS_PER_FRAME = 72 * 1542 + 4 * 774   # trellis steps of the full ensemble: 18 x 4 sub-channel CIFs + 4 FIB groups
VIT_BITS_PER_FRAME = 110592 + 3072          # decoded information bits
FFT_SHIM_NOTE = ("FFT = oracle/fft_shim.cpp (vectorised four-step Stockham, 11 us per 2048 points), not FFTW3f: a real FFTW "
                 "build would make the OFDM stage about 15 % faster")


def _load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def _load_ncu_constants():
    """Per-kernel figures taken from the committed `ncu --set full` summaries of this round (scripts/ncu_constants.py writes the
    file from the reports): DRAM bytes and warp instructions per unit of work.  None when the round has no capture yet."""
    p = os.path.join(ROOT, "profiles", "r2_ncu_constants.json")
    try:
        return json.load(open(p))
    except Exception:
        return {}


_ALL_CPUS = sorted(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else list(range(os.cpu_count() or 1))


def bind_to_gpu_numa(index: int):
    """Pins this process to the CPUs of the NUMA node the GPU hangs off, BEFORE any pinned host buffer is allocated: the pages
    are placed on the node of the allocating thread, and a copy that crosses the socket interconnect shares it with every other
    rank.  Returns a description for the JSON line."""
    info = {"bound": False}
    try:
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(index)
        n_words = (os.cpu_count() + 63) // 64
        try:
            mask = nv.nvmlDeviceGetCpuAffinityWithinScope(h, n_words, nv.NVML_AFFINITY_SCOPE_NODE)
        except Exception:
            mask = nv.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = [64 * w + b for w, word in enumerate(mask) for b in range(64) if (int(word) >> b) & 1]
        allowed = os.sched_getaffinity(0)
        cpus = sorted(set(cpus) & allowed)
        bus = nv.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        node = None
        try:
            node = int(open(f"/sys/bus/pci/devices/{bus[-12:].lower()}/numa_node").read())
        except Exception:
            pass
        info.update({"pci": bus, "node": node, "cpus": len(cpus)})
        if cpus and len(cpus) < len(allowed):
            os.sched_setaffinity(0, cpus)
            info["bound"] = True
    except Exception as e:      # no NVML / no permission: run unbound and say so
        info["error"] = str(e)[:80]
    return info


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons DURING the timed region.  NVML is polled in-process every ~2 ms (an nvidia-smi
    subprocess takes longer than the whole timed region); falls back to the nvidia-smi line of B200_PROFILING.md."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self.stop_flag = False
        self.source = "nvml"
        self.ready = threading.Event()   # set after the first sample: the timed region starts only then

    def _run_nvml(self):
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(self.index)
        self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
        while not self.stop_flag:
            self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
            self.ready.set()
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
            for n, b in bits.items():
                if r & b:
                    self.reasons.add(n)
            time.sleep(0.002)

    def _run_smi(self):
        self.source = "nvidia-smi"
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.ready.set()
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if "Active" in v and "Not" not in v:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.05)

    def run(self):
        try:
            self._run_nvml()
        except Exception:
            self._run_smi()

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_min_mhz": s[0] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s), "source": self.source}


def _sub_array(np, subs):
    return np.array([[sc.start_address, sc.length, int(sc.is_uep), sc.uep_index, sc.eep_level, int(sc.eep_type_b), int(sc.dabplus)]
                     for sc in subs], dtype=np.int32)


def cpu_reference(n_threads: int, frames_per_thread: int, target_seconds: float, full: bool = True):
    """Times the reference's own code (oracle/_ref, unmodified sources) or, if that library is absent, the C port, one
    independent receiver per thread on `n_threads` host threads.  Full workload: OFDM_Demod -> FIC_Decoder + 18 x MSC_Decoder
    (EEP 3-A) + 18 x AAC_Frame_Processor, i.e. what the GPU does per stream.  OFDM workload: OFDM_Demod only.
    Returns (MS/s, kind, sample description, wall seconds, per-core figures or None).  The per-core figures (SURVEY.md section 8(d)) are one
    receiver alone on one core: MS/s and the ms per frame spent in the OFDM demodulator, FIC decoder, MSC decoders and DAB+ processors."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import pyref
    tx = importlib.import_module(PKG + ".synth.dabtx")
    rng = np.random.default_rng(7)
    p = tx.MODES[1]
    subs = tx.default_ensemble()
    use_chain = full and pyref.ref_available() and hasattr(pyref.RefLib.get().L, "ref_time_chain_u8")
    if use_chain:
        ens = tx.EnsembleTx(1, subs, seed=11)
        frames = [ens.next_frame_bits() for _ in range(frames_per_thread)]
    else:
        frames = [rng.integers(0, 2, size=p.nb_frame_bits, dtype=np.uint8) for _ in range(frames_per_thread)]
    iq = tx.ofdm_modulate(frames, 1)
    u8 = tx.to_u8(tx.impair(iq, 15.0, 2.1e-3, 4321, seed=3, tail_samples=2000), 30.0)
    n_samples = u8.size // 2
    what = "OFDM_Demod"
    if use_chain:
        L, kind = pyref.RefLib.get().L, "reference"
        sub_arr = _sub_array(np, subs)
        run = lambda rep: L.ref_time_chain_u8(1, u8, n_samples, BLOCK, rep, sub_arr, len(subs), np.zeros(8, dtype=np.int64))
        what = f"OFDM_Demod + FIC_Decoder + {len(subs)} x (MSC_Decoder + AAC_Frame_Processor)"
    elif pyref.ref_available():
        L, kind = pyref.RefLib.get().L, "reference"
        run = lambda rep: L.ref_time_ofdm_u8(1, u8, n_samples, BLOCK, rep, None)
    else:
        if not pyref.port_available():
            subprocess.check_call(["make", "-s", "port"], cwd=os.path.join(ROOT, "oracle"))
        L, kind = pyref.PortLib.get().L, "port"
        run = lambda rep: L.dabo_time_ofdm_u8(1, u8, n_samples, BLOCK, rep, None)
    t_one = run(1)     # warm-up + calibration of the bounded sample
    t_one = run(1)
    per_core = None
    if use_chain and hasattr(L, "ref_time_chain_split_u8"):
        cnt, split = np.zeros(8, dtype=np.int64), np.zeros(4, dtype=np.float64)
        rep1 = max(1, int(1.5 / max(t_one, 1e-4)))
        t1 = L.ref_time_chain_split_u8(1, u8, n_samples, BLOCK, rep1, sub_arr, len(subs), cnt, split)
        nf = max(int(cnt[0]), 1)
        per_core = {"value": rep1 * n_samples / t1 / 1e6, "unit": "MS/s", "cores": 1, "frames": int(cnt[0]),
                    "ms_per_frame": {"total": 1e3 * t1 / nf, "ofdm": 1e3 * split[0] / nf, "fic": 1e3 * split[1] / nf,
                                     "msc": 1e3 * split[2] / nf, "dabplus_rs": 1e3 * split[3] / nf}}
    repeat = max(2, int(target_seconds / max(t_one, 1e-4)))
    fn = lambda: run(repeat)
    t0 = time.perf_counter()
    ths = [threading.Thread(target=fn) for _ in range(n_threads)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    dt = time.perf_counter() - t0
    msps = n_threads * repeat * n_samples / dt / 1e6
    sample = (f"{n_threads} independent Mode I streams x {repeat}x{frames_per_thread} frames u8 IQ through {what} "
              f"(threads=1 as in the plugin, blocks of {BLOCK}), one receiver per host thread, {dt:.1f} s wall; "
              + (FFT_SHIM_NOTE if kind == "reference" else "C restatement of the chain (oracle/dab_oracle.c)"))
    return msps, kind, sample, dt, per_core


def _workload_name(args):
    return ("full_chain_mode1_" if args.workload == "full" else "ofdm_demod_mode1_") + f"{args.streams}_streams_per_gpu"


def _config(args):
    """The workload both arms measure (BASELINE.json configs[3] per GPU by default)."""
    S, full = args.streams, args.workload == "full"
    return {"workload": _workload_name(args),
            "streams_per_gpu": S, "frame_samples": FRAME_SAMPLES, "process_block": BLOCK, "iq_format": "u8",
            "ensemble": "FIC + 18 x EEP 3-A 48 CU DAB+ sub-channels per stream" if full else "n/a",
            "cache": f"inputs larger than L2: every step reads {S * FRAME_SAMPLES * 2 / 1e6:.0f} MB of IQ last touched {PERIOD_FRAMES} steps ago",
            "snr_db": 15, "cfo": "uniform +-20 kHz", "timing": "uniform lead in [0, 196608)",
            "signal_period_frames": PERIOD_FRAMES, "contexts_per_gpu": max(1, getattr(args, "contexts", 1))}


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores = len(_ALL_CPUS)
    vals, total_dt = [], 0.0
    sample = kind = ""
    for i in range(args.warmup + args.steps):
        msps, kind, sample, dt, per_core = cpu_reference(cores, 20, 4.0, full=args.workload == "full")
        if i >= args.warmup:
            vals.append(msps)
            total_dt += dt
    v = sum(vals) / len(vals)
    line = {
        "impl": "reference", "metric": "dab_mode1_iq_msps", "value": v, "unit": "MS/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total_dt / max(len(vals), 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": _config(args),   # the same keys and values as our arm: the workload is the same, the sample of it is bounded
        "note": "the reference's own CPU code on all host cores, bounded sample of the workload per step; " + FFT_SHIM_NOTE,
        "realtime_streams": v / 2.048,
        "cpu_baseline": {"value": v, "unit": "MS/s", "cores": cores, "kind": kind, "sample": sample, "per_core": per_core},
        "e2e": {"value": v, "unit": "MS/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def spot_check(pkg, tx, np, torch, cyc, subs, local_rank, stream, n_check=3, n_frames=25):
    """The reference chain (oracle/_ref, unmodified sources; the C port has no chain driver) on the first `n_check` streams the
    GPU decoded, `n_frames` frames each, outside every timed region.  The GPU counters of a context that holds just these
    streams must equal the sums of the reference's observer events."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pyref
    if not (pyref.ref_available() and hasattr(pyref.RefLib.get().L, "ref_time_chain_u8")):
        return {"checked": False, "why": "oracle/_ref/libdabref.so not available on this box"}
    L = pyref.RefLib.get().L
    P = cyc.shape[1] // (2 * FRAME_SAMPLES)
    reps = (n_frames + P - 1) // P
    host = cyc[:n_check].repeat(1, reps)[:, :2 * n_frames * FRAME_SAMPLES].contiguous()
    g = pkg.DabGpu(mode=1, max_streams=n_check, device=local_rank, cuda_stream=stream.cuda_stream)
    g.ofdm_attach_device_input(host.data_ptr(), n_frames * FRAME_SAMPLES, n_frames * FRAME_SAMPLES)
    for s in range(n_check):
        g.msc_configure(s, subs)
    for _ in range(n_frames):
        g.ofdm_advance(FRAME_SAMPLES, block_size=BLOCK)
        g.chan_decode()
    c = g.counters()
    g.close()
    h = host.cpu().numpy()
    sub_arr = _sub_array(np, subs)
    tot = np.zeros(8, dtype=np.int64)
    for s in range(n_check):
        cnt = np.zeros(8, dtype=np.int64)
        L.ref_time_chain_u8(1, np.ascontiguousarray(h[s]), n_frames * FRAME_SAMPLES, BLOCK, 1, sub_arr, len(subs), cnt)
        tot += cnt
    ref = {"frames_demodulated": int(tot[0]), "fibs_crc_ok": int(tot[1]), "msc_bytes_decoded": int(tot[2]), "au_ok": int(tot[3]),
           "superframes_ok": int(tot[4]), "superframes_rs_fail": int(tot[5]), "au_crc_fail": int(tot[6])}
    gpu = {k: int(c[k]) for k in ref}
    return {"checked": True, "streams": n_check, "frames_per_stream": n_frames, "identical": gpu == ref, "gpu": gpu, "reference": ref,
            "note": "RS failures come from the superframes that straddle the acquisition: the first logical frames after lock are decoded "
                    "from a time de-interleaver that is only partly filled with real CIFs, in the reference exactly as here"}


def channel_legs(pkg, tx, np, torch, local_rank, stream, n_streams=256, reps=6):
    """BASELINE.json configs[2] / SURVEY.md section 8(d) config 3: the channel decoder alone on `n_streams` streams, soft bits already on the
    device (dabgpu_softbits_push outside the timed region; every stream carries the same coded frames, noisy at 6 dB).  One timed unit =
    dabgpu_chan_decode of one transmission frame of every stream (4 CIFs of every sub-channel + 4 FIB groups)."""
    S = tx.Subchannel
    ensembles = {
        "a_18x_eep_3a_48cu": tx.default_ensemble(),
        "b_eep_mix_1a_to_4b": [S(0, 0, 72, eep_level=0, dabplus=False), S(1, 72, 8, eep_level=1, dabplus=False), S(2, 80, 72, eep_level=1, dabplus=False),
                               S(3, 152, 48, eep_level=2, dabplus=False), S(4, 200, 32, eep_level=3, dabplus=False),
                               S(5, 232, 54, eep_level=0, eep_type_b=True, dabplus=False), S(6, 286, 42, eep_level=1, eep_type_b=True, dabplus=False),
                               S(7, 328, 54, eep_level=2, eep_type_b=True, dabplus=False), S(8, 382, 45, eep_level=3, eep_type_b=True, dabplus=False),
                               S(9, 427, 96, eep_level=2, dabplus=False), S(10, 523, 120, eep_level=1, dabplus=False), S(11, 643, 144, eep_level=0, dabplus=False),
                               S(12, 787, 64, eep_level=3, dabplus=False)],
        "c_uep_rows_0_14_37_63": [S(0, 0, 16, is_uep=True, uep_index=0, dabplus=False), S(1, 16, 32, is_uep=True, uep_index=14, dabplus=False),
                                  S(2, 48, 140, is_uep=True, uep_index=37, dabplus=False), S(3, 188, 416, is_uep=True, uep_index=63, dabplus=False)],
    }
    out = {"streams": n_streams, "unit": "one transmission frame of every stream (4 CIFs of every sub-channel, 4 FIB groups)",
           "input": "coded frames of the synthetic transmitter as int8 soft bits, AWGN 6 dB, resident in the frame ring before the timed region"}
    for name, subs in ensembles.items():
        ens = tx.EnsembleTx(1, subs, seed=21)
        rng = np.random.default_rng(3)
        frames = [tx.hard_to_soft(ens.next_frame_bits(), rng, snr_db=6.0) for _ in range(10)]
        g = pkg.DabGpu(mode=1, max_streams=n_streams, device=local_rank, cuda_stream=stream.cuda_stream)
        for s_ in range(n_streams):
            g.msc_configure(s_, subs)
        batch = [np.ascontiguousarray(np.broadcast_to(f, (n_streams, f.size))) for f in frames]
        for i in range(6):                      # fills the 16-CIF time de-interleavers
            g.softbits_push(batch[i])
            g.chan_decode()
        g.chan_join()
        torch.cuda.synchronize()
        c0 = g.counters()
        total_ms, units = 0.0, 0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for r in range(reps):
            for i in range(4):
                g.softbits_push(batch[(6 + 4 * r + i) % len(batch)])
            torch.cuda.synchronize()
            e0.record(stream)
            for i in range(4):
                g.chan_decode()
            g.chan_join()
            e1.record(stream)
            torch.cuda.synchronize()
            total_ms += e0.elapsed_time(e1)
            units += 4
        c1 = g.counters()
        g.close()
        bits = (c1["msc_bytes_decoded"] - c0["msc_bytes_decoded"]) * 8 + (c1["fibs_total"] - c0["fibs_total"]) * 256
        steps = n_streams * units * (4 * 774 + 4 * sum(sum(n for _, n in sc.segments()) // 4 for sc in subs))
        out[name] = {"sub_channels": len(subs), "capacity_units": sum(sc.length for sc in subs), "ms_per_unit": total_ms / units,
                     "viterbi_mbit_s": bits / (total_ms * 1e-3) / 1e6, "trellis_steps_per_s": steps / (total_ms * 1e-3),
                     "fibs_crc_ok": c1["fibs_crc_ok"] - c0["fibs_crc_ok"], "fibs_total": c1["fibs_total"] - c0["fibs_total"]}
    return out


DUMP_STREAMS, DUMP_SOFT_STREAMS, DUMP_SEED = 512, 16, 2024   # about 44 MB of .npy for the default ensemble
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, np, ctxs, n_subs):
    """Writes what a caller of the timed step receives after its last step, for a fixed seeded sample of the streams (the same
    sample on every run with the same --streams): decoded FIC/MSC bytes as dabgpu_chan_get_fic / dabgpu_chan_get_msc return
    them and the newest soft-bit frame as dabgpu_ofdm_fetch_latest returns it.  Integer outputs are stored as float32 (exact)."""
    per_ctx = ctxs[0].max_streams
    n_all = per_ctx * len(ctxs)
    rng = np.random.default_rng(DUMP_SEED)
    streams = np.sort(rng.choice(n_all, size=min(n_all, DUMP_STREAMS), replace=False))
    soft_streams = np.sort(rng.choice(streams, size=min(streams.size, DUMP_SOFT_STREAMS), replace=False))
    where = lambda s: (ctxs[int(s) // per_ctx], int(s) % per_ctx)
    out = {"streams": streams, "soft_bit_streams": soft_streams}
    latest = [where(s)[0].ofdm_fetch_latest(where(s)[1], 1) for s in soft_streams]
    out["soft_bits"] = np.concatenate([f for f, _ in latest])
    out["soft_bits_produced"] = np.concatenate([p for _, p in latest])
    out["soft_bits"][out["soft_bits_produced"] == 0] = 0      # no frame this step: the staging rows hold stale bytes

    if n_subs:
        fic, fic_ok, msc, msc_valid, status = [], [], [], [], []
        for s in streams:
            g, i = where(s)
            fibs, ok = g.get_fic(i)
            fic.append(fibs)
            fic_ok.append(ok)
            subs = [g.get_msc(i, k) for k in range(n_subs)]
            msc.append(np.concatenate([b for b, _ in subs], axis=1))      # [nb_cifs, bytes of every sub-channel]
            msc_valid.append(np.stack([v for _, v in subs], axis=1))      # [nb_cifs, sub-channels]
            status.append(g.chan_status(i))
        out.update(fic=np.stack(fic), fic_crc_ok=np.stack(fic_ok), msc=np.stack(msc), msc_valid=np.stack(msc_valid),
                   chan_status=np.array(status))
    out = {k: v.astype(np.float32) for k, v in out.items()}
    total = sum(v.nbytes for v in out.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def timed_pass(torch, dist, world, stream, step, K, finish=None, start=None):
    """K steps bracketed by barrier + synchronize, CUDA events on `stream`; returns ms (this rank)."""
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    if start is not None:
        start()           # several contexts: their streams start behind the start event
    for _ in range(K):
        step()
    if finish is not None:
        finish()          # the last channel decode runs on the library's channel stream: make the timing stream wait for it
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=6)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="full", choices=["ofdm", "full"])
    ap.add_argument("--streams", type=int, default=1024)
    ap.add_argument("--e2e-steps", type=int, default=100, help="timed steps of the end-to-end leg (0 skips it: profiling runs only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-spot-check", action="store_true")
    ap.add_argument("--no-ofdm-leg", action="store_true", help="full workload: skip the OFDM-only sub-leg")
    ap.add_argument("--contexts", type=int, default=1, help="device-resident legs: split the streams of a GPU over this many contexts (each with its own CUDA streams)")
    ap.add_argument("--no-channel-leg", action="store_true", help="skip the channel-decode-only sub-legs (BASELINE configs[2])")
    ap.add_argument("--no-c32-leg", action="store_true", help="skip the OFDM-only sub-leg with complex<float> input (256 streams)")
    ap.add_argument("--wc-host", action="store_true", help="e2e: write-combined pinned memory for the IQ the host feeds in")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps of the main leg, write what its last step computed "
                                                           "(seeded sample of rank 0's streams) to DIR/<name>.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    args.warmup = max(args.warmup, 6)     # >= 5 frames: the time de-interleavers emit nothing before 16 CIFs

    numa = bind_to_gpu_numa(local_rank)   # before CUDA / pinned allocations

    import numpy as np
    import torch
    import torch.distributed as dist

    pkg = importlib.import_module(PKG)
    synth = importlib.import_module(PKG + ".synth.gpusynth")
    tx = importlib.import_module(PKG + ".synth.dabtx")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the DAB path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    S, K, W = args.streams, args.steps, args.warmup
    full = args.workload == "full"
    subs = tx.default_ensemble()
    # two distinct periodic coded ensembles (FIC + 18 x EEP 3-A DAB+ sub-channels), shared by the streams with different channels
    payload = np.stack([tx.periodic_frames(1, subs, seed=1000 * (rank + 1) + u, period_frames=PERIOD_FRAMES) for u in range(2)])
    # the job is world * S streams; stream s belongs to rank s mod world (shard.py) -- no data-path collective, every rank builds
    # and decodes only its own streams (the channel of a stream is seeded by the first global id of the rank's share)
    shard = importlib.import_module(PKG + ".shard")
    my_streams = shard.streams_for_rank(world * S, rank, world)
    assert len(my_streams) == S and all(shard.owner_of(s_, world) == rank for s_ in my_streams)
    cyc, _, _ = synth.make_cyclic_streams_u8(S, payload, mode=1, seed0=1 + my_streams[0], snr_db=15.0, device=str(dev))
    n_frames = W + 2 * K + 2          # K timed steps for `value`, K more with per-kernel CUDA events for the roofline
    reps = (n_frames + PERIOD_FRAMES - 1) // PERIOD_FRAMES
    iq = cyc.repeat(1, reps)
    total_samples = iq.shape[1] // 2
    torch.cuda.synchronize()

    # a non-default stream: the library launches every kernel on it and torch.cuda.Event times that same stream
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)

    NCTX = max(1, args.contexts)
    assert S % NCTX == 0

    class CtxGroup:
        """`NCTX` contexts of S / NCTX streams each on this GPU, every one with its own main CUDA stream (and, inside the library,
        its own channel stream): the step of one context overlaps the step of the others.  With one context this is the plain API."""

        def __init__(self, with_chan, n_streams=None):
            self.with_chan = with_chan
            self.n = (n_streams or S) // NCTX
            self.streams = [stream] if NCTX == 1 else [torch.cuda.Stream(dev) for _ in range(NCTX)]
            self.ctxs = []
            self.done = [torch.cuda.Event() for _ in range(NCTX)]
            for c in range(NCTX):
                g = pkg.DabGpu(mode=1, max_streams=self.n, device=local_rank, cuda_stream=self.streams[c].cuda_stream)
                g.ofdm_attach_device_input(iq.data_ptr() + c * self.n * iq.stride(0), total_samples, total_samples)
                if with_chan:
                    for s in range(self.n):
                        g.msc_configure(s, subs)
                self.ctxs.append(g)

        def fork(self):      # the contexts' streams start after everything queued on the timing stream so far
            if NCTX > 1:
                ev = torch.cuda.Event()
                ev.record(stream)
                for st in self.streams:
                    st.wait_event(ev)

        def step(self):
            for g in self.ctxs:
                g.ofdm_advance(FRAME_SAMPLES, block_size=BLOCK)
                if self.with_chan:
                    g.chan_decode()

        def join(self):      # the timing stream waits for every context (its channel stream included)
            for c, g in enumerate(self.ctxs):
                if self.with_chan:
                    g.chan_join()
                if NCTX > 1:
                    self.done[c].record(self.streams[c])
                    stream.wait_event(self.done[c])

        def counters(self):
            cs = [g.counters() for g in self.ctxs]
            return {k: sum(c[k] for c in cs) for k in cs[0]}

        @property
        def launch_count(self):
            return sum(g.launch_count for g in self.ctxs)

        def profile_enable(self, on):
            for g in self.ctxs:
                g.profile_enable(on)

        def profile_read(self):
            ps = [g.profile_read() for g in self.ctxs]
            return {k: {"ms": sum(p_[k]["ms"] for p_ in ps), "launches": sum(p_[k]["launches"] for p_ in ps)} for k in ps[0]}

        def close(self):
            for g in self.ctxs:
                g.close()

    class C32Group(CtxGroup):      # one context fed complex<float>: the plugin's own input format (src/dab_module.cpp:20-28)
        def __init__(self, c32):
            self.with_chan, self.n, self.streams, self.done = False, c32.shape[0], [stream], []
            g = pkg.DabGpu(mode=1, max_streams=c32.shape[0], device=local_rank, iq_format=pkg.IQ_C32, cuda_stream=stream.cuda_stream)
            g.ofdm_attach_device_input(c32.data_ptr(), c32.shape[1] // 2, c32.shape[1] // 2)
            self.ctxs = [g]

        def fork(self):
            pass

        def join(self):
            pass

    def run_leg(with_chan, K=K, c32=None, n_streams=None, dump_dir=None):
        """W warm-up steps, K timed steps (device-resident), K profiled steps.  Returns a dict of raw measurements.
        dump_dir: write the outputs of the last timed step there (dump_outputs) before the profiled steps change them."""
        g = CtxGroup(with_chan, n_streams) if c32 is None else C32Group(c32)

        def step():
            g.step()

        g.fork()
        for _ in range(W):
            step()
        g.join()
        torch.cuda.synchronize()
        c0 = g.counters()
        launches0 = g.launch_count
        ms = timed_pass(torch, dist, world, stream, step, K, finish=g.join, start=g.fork)
        c1 = g.counters()
        launches = g.launch_count - launches0
        if dump_dir and rank == 0:
            dump_outputs(dump_dir, np, g.ctxs, len(subs) if with_chan else 0)
        # second pass with CUDA events around every kernel launch (dabgpu_profile_*): per-kernel times for the roofline.  The
        # library keeps the channel decode on the main stream while profiling, so this pass is slower than the one above.
        g.profile_enable(True)
        ms_prof = timed_pass(torch, dist, world, stream, step, K, finish=g.join, start=g.fork)
        prof = g.profile_read()
        g.profile_enable(False)
        c2 = g.counters()
        g.close()
        return {"ms": ms, "ms_prof": ms_prof, "prof": prof, "c0": c0, "c1": c1, "c2": c2, "launches": launches}

    sampler = ClockSampler(local_rank)
    sampler.start()
    sampler.ready.wait(timeout=20)   # NVML initialisation on a fresh box can take longer than the whole timed region
    sampler.samples.clear()          # keep only what is sampled while the kernels run
    main_leg = run_leg(full, dump_dir=args.dump_outputs)
    sampler.stop_flag = True
    sampler.join(timeout=2)
    clocks = sampler.summary()
    ms, prof = main_leg["ms"], main_leg["prof"]
    c0, c1, c2 = main_leg["c0"], main_leg["c1"], main_leg["c2"]

    def allmax(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    ms_max = allmax(ms)
    frames_all = allsum(c1["frames_demodulated"] - c0["frames_demodulated"])
    # whole-job throughput: samples actually consumed by all ranks / max time (every stream advances one frame per step)
    value = world * S * FRAME_SAMPLES * K / (ms_max * 1e-3) / 1e6

    # ---- end to end through the C ABI with HOST buffers: dabgpu_submit / dabgpu_wait, two tickets in flight ----
    # every step copies that step's u8 IQ from pinned host memory (H2D), runs the kernels and copies the step's results back
    # (D2H): the decoded FIC/MSC bytes for the full chain, the soft-bit frames for the OFDM workload.  The host buffer holds one
    # period of the transmission and is walked cyclically.
    Ke = args.e2e_steps
    e2e_value = e2e_ms_max = None
    n_prod, d2h_bytes, h2d_bytes, e2e_counters = 0, 0, S * FRAME_SAMPLES * 2, {}
    if Ke > 0:
        P = pkg.get_params(1)
        hb = pkg.HostBuffer(S * 2 * PERIOD_FRAMES * FRAME_SAMPLES, write_combined=args.wc_host)
        h_np = hb.array.reshape(S, 2 * PERIOD_FRAMES * FRAME_SAMPLES)
        torch.from_numpy(h_np).copy_(cyc)
        D = pkg.PIPELINE_DEPTH
        if full:
            outs = [dict(msc_host=torch.empty((S, P.nb_cifs, pkg.CIF_OUT_STRIDE), dtype=torch.uint8).pin_memory(),
                         fic_host=torch.empty((S, P.nb_cifs, pkg.FIC_GROUP_STRIDE), dtype=torch.uint8).pin_memory(),
                         fic_crc_host=torch.empty((S, P.nb_cifs, 4), dtype=torch.uint8).pin_memory(),
                         msc_valid_host=torch.empty((S, P.nb_cifs, 64), dtype=torch.uint8).pin_memory(),
                         chan_status_host=torch.zeros((S, 2), dtype=torch.int32).pin_memory()) for _ in range(D)]
        else:
            outs = [dict(frames_host=torch.empty((S, P.nb_frame_bits), dtype=torch.int8).pin_memory(),
                         produced_host=torch.zeros(S, dtype=torch.uint8).pin_memory()) for _ in range(D)]
        d2h_bytes = sum(t.numel() * t.element_size() for t in outs[0].values())
        h2d_bytes = S * FRAME_SAMPLES * 2
        g2 = pkg.DabGpu(mode=1, max_streams=S, device=local_rank, cuda_stream=stream.cuda_stream)
        if full:
            for s in range(S):
                g2.msc_configure(s, subs)
        tickets = {}
        n_prod = 0

        def e2e_submit(i):
            o = outs[i % D]
            view = h_np[:, 2 * (i % PERIOD_FRAMES) * FRAME_SAMPLES: 2 * ((i % PERIOD_FRAMES) + 1) * FRAME_SAMPLES]
            tickets[i] = g2.submit(view.ctypes.data, h_np.strides[0], FRAME_SAMPLES, block_size=BLOCK, run_chan_decode=full,
                                   **{k: v.data_ptr() for k, v in o.items()})

        def e2e_retire(i):
            g2.wait(tickets.pop(i))
            o = outs[i % D]
            return int(o["chan_status_host"][:, 0].sum()) if full else int(o["produced_host"].sum())

        for i in range(W):
            e2e_submit(i)
            e2e_retire(i)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(stream)
        for i in range(W, W + Ke):
            if i - D >= W:
                n_prod += e2e_retire(i - D)
            e2e_submit(i)
        for i in range(max(W, W + Ke - D), W + Ke):
            n_prod += e2e_retire(i)
        e1.record(stream)
        torch.cuda.synchronize()
        e2e_ms = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)
        e2e_ms_max = allmax(e2e_ms)
        e2e_value = world * S * FRAME_SAMPLES * Ke / (e2e_ms_max * 1e-3) / 1e6
        e2e_counters = g2.counters()
        g2.close()
        hb.close()

    # ---- roofline of the dominant kernel of the step ----
    peak, peak_src = _load_peaks()
    ncu = _load_ncu_constants()
    frames_prof = c2["frames_demodulated"] - c1["frames_demodulated"]
    frames_chan_prof = c2["frames_channel_decoded"] - c1["frames_channel_decoded"]
    ms_prof = main_leg["ms_prof"]
    sm_hz = (clocks["sm_mhz"] or 1965.0) * 1e6
    n_sms = torch.cuda.get_device_properties(dev).multi_processor_count

    def roofline_ofdm(prof_, frames_, ms_prof_, c32=False, n_streams=None):
        t = prof_["ofdm_demod"]["ms"]
        n = prof_["ofdm_demod"]["launches"]
        alg = OFDM_ALG_BYTES_C32 if c32 else OFDM_ALG_BYTES
        ach = frames_ * alg / (t * 1e-3) / 1e9 if t > 0 else 0.0
        k = ncu.get("k_ofdm_demod2", {})
        return {"kernel": "k_ofdm_demod2<2048,c32>" if c32 else "k_ofdm_demod2<2048,u8>", "bound": "hbm", "achieved": ach, "peak": peak,
                "unit": "GB/s", "frac": ach / peak,
                # per launch that has work: one frame of every stream (the launch count also holds the empty launches of a step)
                "traffic": k["dram_bytes_per_frame"] * (n_streams or S) if ("dram_bytes_per_frame" in k and not c32) else None,
                "algorithmic_bytes_per_frame": alg, "frames_in_profiled_pass": frames_, "kernel_ms_total": t, "kernel_launches": n,
                "kernel_share_of_step": t / ms_prof_ if ms_prof_ > 0 else None,
                "issue": {"warp_inst_per_sample": k.get("warp_inst_per_sample"), "issue_active_pct": k.get("issue_active_pct"),
                          # SURVEY.md section 8(d): ~17.7 M floating-point operations per Mode I frame (FFT 8.56, PLL 6.9, sync 0.56, CP 0.31, DQPSK 1.4)
                          "fp32_tflops_algorithmic": frames_ * OFDM_ALG_FLOP / (t * 1e-3) / 1e12 if t > 0 else None,
                          "source": k.get("source")},
                "note": ("c32 input (the plugin's own format, 8 B/sample): " if c32 else "u8 input (2 B/sample): ") +
                        "this kernel is FP32-issue bound (~100 instructions per sample), not HBM bound; see DESIGN.md"}

    def roofline_viterbi():
        t = prof["viterbi"]["ms"]
        n = prof["viterbi"]["launches"]
        ach = frames_chan_prof * VIT_ALG_BYTES / (t * 1e-3) / 1e9 if t > 0 else 0.0
        k = ncu.get("k_viterbi_lanes", {})
        steps = frames_chan_prof * VIT_STEPS_PER_FRAME
        alu = k.get("alu_pipe_warp_inst_per_32_steps")
        # ALU-pipe issue rate measured on this part: 0.5 warp instructions per clock and SM sub-partition (profiles/r1e_micro_pipe_rates.txt)
        alu_frac = (steps / 32.0 * alu) / (n_sms * 4 * 0.5 * sm_hz * t * 1e-3) if (alu and t > 0) else None
        return {"kernel": "k_viterbi_lanes", "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": k["dram_bytes_per_frame"] * frames_chan_prof / max(n, 1) if "dram_bytes_per_frame" in k else None,
                "algorithmic_bytes_per_frame": VIT_ALG_BYTES, "frames_in_profiled_pass": frames_chan_prof, "kernel_ms_total": t,
                "kernel_launches": n, "kernel_share_of_step": t / ms_prof if ms_prof > 0 else None,
                "issue": {"bound": "integer ALU pipe (VIADDMNMX/VIMNMX.U16x2 at 0.5 warp-instr/clk/sub-partition)",
                          "acs_per_s": steps * 64 / (t * 1e-3) if t > 0 else None,
                          "decoded_mbit_s": frames_chan_prof * VIT_BITS_PER_FRAME / (t * 1e-3) / 1e6 if t > 0 else None,
                          "alu_pipe_frac": alu_frac, "alu_pipe_warp_inst_per_32_steps": alu,
                          "warp_inst_per_32_steps": k.get("warp_inst_per_32_steps"), "source": k.get("source")},
                "note": "the contract's HBM figure is kept for comparability; this kernel is bound by the integer ALU pipe, see `issue`"}

    roofs = {"ofdm_demod": roofline_ofdm(prof, frames_prof, ms_prof)}
    if full:
        roofs["viterbi"] = roofline_viterbi()
    dominant = max(roofs, key=lambda k_: roofs[k_]["kernel_ms_total"])
    roofline = dict(roofs[dominant])
    roofline["peak_source"] = f"{peak_src} (MEASURED_PEAKS.json hbm_gbs)" if peak_src == "measured" else "fallback 6.65 TB/s (B200_PROFILING.md)"
    roofline["profiled_pass_ms_per_step"] = ms_prof / K
    roofline["other_kernels"] = {k_: {f: v[f] for f in ("kernel", "achieved", "frac", "kernel_ms_total", "kernel_share_of_step")}
                                 for k_, v in roofs.items() if k_ != dominant}

    bits = lambda a, b: (b["msc_bytes_decoded"] - a["msc_bytes_decoded"]) * 8 + (b["fibs_total"] - a["fibs_total"]) * 256
    line = {
        "metric": "dab_mode1_iq_msps", "value": value, "unit": "MS/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (OFDM) / u16 (Viterbi) / u8 (RS)",
        "data": "synthetic",
        "config": _config(args),
        "realtime_streams": value / 2.048,
        "frames_demodulated": frames_all,
        "e2e": None if Ke <= 0 else {"value": e2e_value, "unit": "MS/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                "steps": Ke, "ms_per_step": e2e_ms_max / Ke, "frames_returned": n_prod,
                "h2d_gb_s_per_gpu": h2d_bytes / (e2e_ms_max / Ke * 1e-3) / 1e9, "d2h_gb_s_per_gpu": d2h_bytes / (e2e_ms_max / Ke * 1e-3) / 1e9,
                "realtime_streams": e2e_value / 2.048,
                "limit": "PCIe H2D of the u8 IQ (2 B/sample is the smallest input format the reference accepts)",
                "host_memory": ("write-combined " if args.wc_host else "") + "pinned (dabgpu_host_alloc), allocated after binding to the GPU's NUMA node",
                "api": "dabgpu_submit/dabgpu_wait, 2 tickets in flight"},
        "numa": numa,
        "gpu_launches": int(main_leg["launches"]),
        "kernel_ms": {k: v["ms"] for k, v in prof.items()},
        "roofline": roofline,
        "clocks": clocks,
    }
    if full:
        line["viterbi_mbit_s"] = bits(c1, c2) / ((prof["viterbi"]["ms"] + prof["chan_misc"]["ms"]) * 1e-3) / 1e6
        line["viterbi_mbit_s_whole_chain"] = bits(c0, c1) / (ms * 1e-3) / 1e6
        line["counters"] = {k: c1[k] - c0[k] for k in c1}
        if line["e2e"] is not None:
            line["e2e"]["counters"] = e2e_counters
        if not args.no_ofdm_leg:
            leg = run_leg(False)
            fr = leg["c2"]["frames_demodulated"] - leg["c1"]["frames_demodulated"]
            ms_o = allmax(leg["ms"])
            line["ofdm_only"] = {"workload": f"ofdm_demod_mode1_{S}_streams_per_gpu", "ms_per_step": ms_o / K,
                                 "iq_msps": world * S * FRAME_SAMPLES * K / (ms_o * 1e-3) / 1e6, "kernel_ms": {k: v["ms"] for k, v in leg["prof"].items()},
                                 "roofline": roofline_ofdm(leg["prof"], fr, leg["ms_prof"])}
    if not args.no_ofdm_leg and S > 256 and NCTX == 1:
        # BASELINE.json configs[1] as it is written: OFDM demodulation only, 256 Mode I streams on one GPU
        leg = run_leg(False, n_streams=256)
        fr = leg["c2"]["frames_demodulated"] - leg["c1"]["frames_demodulated"]
        ms_o = allmax(leg["ms"])
        line["ofdm_only_256"] = {"workload": "ofdm_demod_mode1_256_streams_per_gpu", "ms_per_step": ms_o / K,
                                 "iq_msps": world * 256 * FRAME_SAMPLES * K / (ms_o * 1e-3) / 1e6, "kernel_ms": {k: v["ms"] for k, v in leg["prof"].items()},
                                 "roofline": roofline_ofdm(leg["prof"], fr, leg["ms_prof"], n_streams=256)}
    if full and not args.no_channel_leg and rank == 0:
        # BASELINE.json configs[2]: MSC channel decode alone (time de-interleave + de-puncture + Viterbi + descramble, DAB+ RS where the
        # sub-channel carries it) for the protection profiles of SURVEY.md section 8(d) config 3, 256 streams, soft bits pushed beforehand
        try:
            line["channel_decode"] = channel_legs(pkg, tx, np, torch, local_rank, stream)
        except Exception as e:
            line["channel_decode"] = {"error": str(e)[:200]}
    if not args.no_c32_leg:
        # the same OFDM workload fed as complex<float> (what SDR++ hands the plugin): 9.17 instead of 3.17 algorithmic bytes per sample
        Sc, Kc = min(S, 256), min(K, 20)
        reps_c = (W + 2 * Kc + 2 + PERIOD_FRAMES - 1) // PERIOD_FRAMES
        c32 = torch.empty((Sc, 2 * reps_c * PERIOD_FRAMES * FRAME_SAMPLES), dtype=torch.float32, device=dev)
        for s_ in range(Sc):        # the conversion of app_iq_readers.h:23-43: (u8 - 127.5) * (1 / 127.5)
            c32[s_] = ((cyc[s_].to(torch.float32) - 127.5) * np.float32(1.0 / 127.5)).repeat(reps_c)
        torch.cuda.synchronize()
        leg = run_leg(False, K=Kc, c32=c32)
        fr = leg["c2"]["frames_demodulated"] - leg["c1"]["frames_demodulated"]
        ms_c = allmax(leg["ms"])
        line["ofdm_only_c32"] = {"workload": f"ofdm_demod_mode1_{Sc}_streams_per_gpu_c32_input", "steps": Kc, "ms_per_step": ms_c / Kc,
                                 "iq_msps": world * Sc * FRAME_SAMPLES * Kc / (ms_c * 1e-3) / 1e6,
                                 "kernel_ms": {k: v["ms"] for k, v in leg["prof"].items()},
                                 "roofline": roofline_ofdm(leg["prof"], fr, leg["ms_prof"], c32=True)}
        del c32
    # cuFFT as the stated comparison point of the FFT stage: a batched 2048-point C2C transform of as many symbols as one step
    # demodulates, c32 in HBM -> c32 in HBM (torch.fft = cuFFT), against the whole fused kernel that also does PLL, CP
    # correlation, DQPSK, de-interleave and quantisation and moves 2 + 1.17 instead of 8 + 8 bytes per sample
    if rank == 0:
        try:
            nsym = min(S, 256) * 76
            x = torch.randn((nsym, 2048), dtype=torch.complex64, device=dev)
            for _ in range(3):
                torch.fft.fft(x)
            torch.cuda.synchronize()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record(stream)
            for _ in range(10):
                y = torch.fft.fft(x)
            f1.record(stream)
            torch.cuda.synchronize()
            cufft_ms = f0.elapsed_time(f1) / 10
            d = roofs["ofdm_demod"]
            ours_ms = d["kernel_ms_total"] / max(d["frames_in_profiled_pass"], 1) * min(S, 256)
            line["cufft_comparison"] = {"what": f"cuFFT C2C 2048 x {nsym} (the FFTs of {min(S, 256)} frames), c32 HBM -> c32 HBM, comparison only",
                                        "cufft_ms": cufft_ms, "k_ofdm_demod2_ms_same_frames": ours_ms,
                                        "note": "the fused kernel runs one extra FFT per 15-symbol chunk, the PLL, CP correlation, DQPSK, "
                                                "de-interleave and quantisation in that time and never writes a spectrum to HBM"}
            del x, y
        except Exception as e:
            line["cufft_comparison"] = {"error": str(e)[:120]}
    if rank == 0 and full and not args.no_spot_check:
        try:
            line["spot_check"] = spot_check(pkg, tx, np, torch, cyc, subs, local_rank, stream)
        except Exception as e:
            line["spot_check"] = {"checked": False, "why": str(e)[:160]}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        if hasattr(os, "sched_setaffinity"):
            os.sched_setaffinity(0, _ALL_CPUS)      # the CPU arm uses every host core again
        cores = len(_ALL_CPUS)
        v, kind, sample, _, per_core = cpu_reference(cores, 20, 12.0, full=full)
        line["cpu_baseline"] = {"value": v, "unit": "MS/s", "cores": cores, "kind": kind, "sample": sample, "per_core": per_core}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
