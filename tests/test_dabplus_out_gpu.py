"""Batched DAB+ output on the GPU (k_dabplus_pack): dabgpu_chan_get_dabplus_all, dabgpu_submit_ex and dabgpu_wideband_submit_ex.

Bar: the log of every (stream, sub-channel) is byte-identical to dabgpu_chan_get_dabplus_events after the same decode and to
the oracle's observer log; nothing outside the requested streams is reported and every other index entry has length 0; each
pipelined ticket delivers its own decode's output with two tickets in flight; refused requests leave the context as it was."""
import ctypes as C
import dataclasses
import importlib

import numpy as np
import pytest

import dabplus_cases as dc
from test_dabplus_gpu import _aac, _batched_subs, _counts, _delta

pytestmark = pytest.mark.gpu

BLOCK = 65536
FRACTIONS = (0.3, 1.0, 0.7, 1.4)   # pipelined ticket sizes in frames of input


def raw_all(dab, g, first, n):
    """dabgpu_chan_get_dabplus_all into poisoned buffers: (log, index [n][max_subchannels][2])"""
    log = np.full(max(g.dabplus_out_bound(first, n), 1), 0xA5, dtype=np.uint8)
    index = np.full((n, g.max_subchannels, 2), -7, dtype=np.int32)
    out = dab.DabPlusOut(log.ctypes.data, log.size, index.ctypes.data)
    dab._check(g.L.dabgpu_chan_get_dabplus_all(g.h, first, n, C.byref(out)))
    return log, index


def check_packed(dab, pyref, g, first, n, log, index, want, tag):
    """log / index of streams [first, first + n) against want = {(stream, sub): log}; entries missing from want must be empty"""
    index = np.asarray(index).reshape(n, g.max_subchannels, 2)
    off, ln = index[..., 0].astype(np.int64), index[..., 1].astype(np.int64)
    assert (ln >= 0).all() and (off[ln > 0] % 4 == 0).all() and (off + ln <= log.size).all(), f"{tag}: index out of the log"
    got = dab.split_dabplus(log, index, first, g.max_subchannels)
    assert set(got) == {key for key, v in want.items() if v}, f"{tag}: non-empty entries {sorted(set(got) ^ {k for k, v in want.items() if v})} differ"
    for key, v in got.items():
        assert v == want[key], f"{tag}: {key}: {[e[:5] for e in pyref.parse_event_log(v)]} != {[e[:5] for e in pyref.parse_event_log(want[key])]}"
    return got


def fake_superframes(tx, pyref):
    """tx.build_superframe stand-in cycling through test_dabplus_gpu's cases per bitrate: every AU layout, the longest last AU,
    AU CRC failures, uncorrectable codewords, fire-code failures, 2 115-byte AUs and corrected byte errors"""
    rs = pyref.PortRS()
    count = {}

    def fake(bitrate_kbps, rng, **_):
        N = bitrate_kbps // 8
        k = count[N] = count.get(N, -1) + 1
        dac_rate, sbr = dc.LAYOUTS[(k // 6) % 4]
        n_aus = dc.N_AUS[(dac_rate, sbr)]
        kw = dict(dac_rate=dac_rate, sbr=sbr, mpeg=(0, 1, 2, 7, 3)[k % 5])
        case = k % 6
        if case == 1:
            return dc.build(tx, rng, N, starts=dc.split_starts(N, n_aus, [0] * (n_aus - 1)), **kw).sf
        if case == 2:
            return dc.build(tx, rng, N, bad_crc=(k % n_aus,), **kw).sf
        if case == 3:
            s = dc.build(tx, rng, N, **kw)
            while True:
                t = s.with_errors(dc.cw_errors(rng, N - 1, 7), "")
                if rs.decode(t.sf[N - 1:120 * N:N])[0] < 0:
                    return t.sf
        if case == 4:
            return dc.build(tx, rng, N, bad_fire=True, **kw).sf
        if case == 5 and dc.header_len(n_aus) + 2117 + k % 3 + 2 * (n_aus - 1) <= 110 * N:
            return dc.build(tx, rng, N, starts=dc.split_starts(N, n_aus, [2115 + k % 3] + [0] * (n_aus - 2)), **kw).sf
        s = dc.build(tx, rng, N, **kw)
        return s.with_errors(sum((dc.cw_errors(rng, cw, 5) for cw in range(0, N, 3)), []), "").sf

    return fake


class OracleLogs:
    """The oracle's AAC_Frame_Processor per (stream, sub index), fed the MSC bytes the GPU decoded; `last` holds the log of
    the last decode that covered each stream (what the getters report)."""

    def __init__(self, pyref):
        self.pyref, self.aacs, self.last, self.events = pyref, {}, {}, []

    def attach(self, s, k):
        self.aacs[(s, k)] = _aac(self.pyref)

    def detach(self, s, k):
        self.aacs.pop((s, k), None)
        self.last.pop((s, k), None)

    def decoded(self, g, first, n, tag):
        """after chan_decode(first, n): oracle logs of those streams, each equal to the per-sub getter"""
        for (s, k), aac in self.aacs.items():
            if not first <= s < first + n:
                continue
            exp = []
            if g.chan_status(s)[0]:
                out, valid = g.get_msc(s, k)
                for c in range(g.P.nb_cifs):
                    if valid[c]:
                        exp += aac.process(out[c])
            self.events += exp
            self.last[(s, k)] = dc.event_log(exp)
            assert g.get_dabplus_events(s, k) == self.last[(s, k)], f"{tag}: stream {s} sub-channel {k}: per-sub getter != oracle"

    def want(self, first, n):
        return {key: v for key, v in self.last.items() if first <= key[0] < first + n}


def run_sync(dab, tx, pyref, mode, stream_subs, n_frames, schedule, monkeypatch):
    """softbits_push -> chan_decode -> get_dabplus_all over several ranges; schedule[f] = ((push first, n), (decode first, n))"""
    monkeypatch.setattr(tx, "build_superframe", fake_superframes(tx, pyref))
    S = len(stream_subs)
    enss = [tx.EnsembleTx(mode, stream_subs[s], seed=300 + 7 * s) for s in range(S)]
    g = dab.DabGpu(mode=mode, max_streams=S)
    ref = OracleLogs(pyref)
    for s in range(S):
        g.msc_configure(s, stream_subs[s])
        for k, sc in enumerate(stream_subs[s]):
            if sc.dabplus:
                ref.attach(s, k)
    c0 = g.counters()
    for f in range(n_frames):
        (pf, pn), (df, dn) = schedule.get(f, ((0, S), (0, S)))
        g.softbits_push(np.stack([tx.hard_to_soft(enss[s].next_frame_bits()) for s in range(pf, pf + pn)]), first_stream=pf)
        g.chan_decode(df, dn)
        ref.decoded(g, df, dn, f"mode {mode} frame {f}")
        for first, n in sorted({(0, S), (df, dn)} | {(s, 1) for s in range(S)} | ({(1, S - 1)} if S > 1 else set())):
            log, index = raw_all(dab, g, first, n)
            got = check_packed(dab, pyref, g, first, n, log, index, ref.want(first, n), f"mode {mode} frame {f} streams [{first}, {first + n})")
            if (first, n) == (0, S):
                assert g.get_dabplus_all(first, n) == got
    assert _delta(g, c0) == _counts(pyref, ref.events)
    g.close()
    return ref.events


def _mixed_subs(tx, subs, plain):
    return [dataclasses.replace(sc, dabplus=False) if i in plain else sc for i, sc in enumerate(subs)]


def test_sync_batch_every_case_partial_ranges(gpu_ctx, tx, pyref, monkeypatch):
    """three streams with 13 sub-channels (two of them not DAB+; the last stream has only 7), superframes replaced by the
    oracle-checked error cases; decode calls over streams 1-2, stream 0 only, and all three with stream 0 given no frame"""
    subs = _mixed_subs(tx, _batched_subs(tx), (3, 9))
    schedule = {12: ((1, 2), (1, 2)), 21: ((0, 1), (0, 1)), 25: ((1, 2), (0, 3)), 26: ((1, 2), (0, 3))}
    events = run_sync(gpu_ctx, tx, pyref, 1, [subs, subs, subs[:7]], 30, schedule, monkeypatch)
    kinds = {e[0] for e in events}
    assert kinds == {pyref.EV_HEADER, pyref.EV_AU, pyref.EV_AU_CRC_ERROR, pyref.EV_RS_ERROR, pyref.EV_FIRECODE_ERROR}, kinds
    assert any(e[0] == pyref.EV_AU and len(e[5]) >= 2115 for e in events), "no AU of 2115 bytes or more"


@pytest.mark.parametrize("mode", [2, 4])
def test_sync_batch_modes_2_and_4(gpu_ctx, tx, pyref, monkeypatch, mode):
    """1 and 2 CIFs per frame: most calls deliver no AU and every superframe spans several decode calls"""
    subs = _mixed_subs(tx, _batched_subs(tx)[:8], (2,))
    n_frames = 60 if mode == 2 else 40
    events = run_sync(gpu_ctx, tx, pyref, mode, [subs, subs[:5]], n_frames, {17: ((1, 1), (0, 2))}, monkeypatch)
    assert sum(e[0] == pyref.EV_AU for e in events) > 0 and sum(e[0] == pyref.EV_HEADER for e in events) >= 8


def test_sync_batch_follows_add_and_remove(gpu_ctx, tx, pyref):
    """msc_add_subchannel / msc_remove_subchannel between decodes: the index follows the new tables and the bound with them"""
    dab = gpu_ctx
    subs = _mixed_subs(tx, _batched_subs(tx)[:9], (4,))
    enss = [tx.EnsembleTx(1, subs, seed=90 + s) for s in range(2)]
    g = dab.DabGpu(mode=1, max_streams=2)
    ref = OracleLogs(pyref)
    table = [[], []]   # per stream: the Subchannel of each sub index, None once removed

    def add(s, sc):
        k = g.msc_add_subchannel(s, sc)
        assert k == len(table[s])
        table[s].append(sc)
        if sc.dabplus:
            ref.attach(s, k)

    for s in range(2):
        for sc in subs[:3]:
            add(s, sc)
    bounds = [g.dabplus_out_bound(0, 2)]
    for f in range(24):
        if f == 6:
            for sc in subs[3:7]:
                add(0, sc)
            bounds.append(g.dabplus_out_bound(0, 2))
            assert bounds[-1] > bounds[-2]
        if f == 12:
            for s, k in ((1, 1), (0, 5)):
                g.msc_remove_subchannel(s, k)
                table[s][k] = None
                ref.detach(s, k)
            bounds.append(g.dabplus_out_bound(0, 2))
            assert bounds[-1] < bounds[-2]
        if f == 16:
            add(1, subs[8])
            bounds.append(g.dabplus_out_bound(0, 2))
            assert bounds[-1] > bounds[-2]
        for s in range(2):   # the contract's argument: at most 7 events and 5 CIFs of payload per DAB+ sub-channel
            live = [sc for sc in table[s] if sc is not None and sc.dabplus]
            assert g.dabplus_out_bound(s, 1) >= sum(7 * 24 + 5 * sc.frame_bytes for sc in live)
            assert (g.dabplus_out_bound(s, 1) == 0) == (not live)
        assert g.dabplus_out_bound(0, 1) + g.dabplus_out_bound(1, 1) == g.dabplus_out_bound(0, 2)
        g.softbits_push(np.stack([tx.hard_to_soft(e.next_frame_bits()) for e in enss]))
        g.chan_decode()
        ref.decoded(g, 0, 2, f"frame {f}")
        for first, n in ((0, 2), (0, 1), (1, 1)):
            log, index = raw_all(dab, g, first, n)
            check_packed(dab, pyref, g, first, n, log, index, ref.want(first, n), f"frame {f} streams [{first}, {first + n})")
    assert sum(e[0] == pyref.EV_AU for e in ref.events) > 0
    g.close()


# ---- pipelined -----------------------------------------------------------------------------------------------------------------
def narrowband_iq(tx, subs, n_streams, n_frames, seed):
    recs = []
    for s in range(n_streams):
        ens = tx.EnsembleTx(1, subs, seed=seed + s)
        iq = tx.ofdm_modulate([ens.next_frame_bits() for _ in range(n_frames)], 1)
        recs.append(tx.to_u8(tx.impair(iq, 18.0, (1.5 - 3 * s) * 1e-3, 777 + 5000 * s, seed=seed + s, tail_samples=3000), 30.0))
    n = min(r.size for r in recs)
    return np.stack([r[:n] for r in recs])


class TicketOut:
    """pinned DAB+ log + index and chan_status / msc arenas of one ticket"""

    def __init__(self, dab, g, first, n):
        self.n, self.g = n, g
        self.log = dab.HostBuffer(max(g.dabplus_out_bound(first, n), 1))
        self.index = dab.HostBuffer(n * g.max_subchannels * 8)
        self.status = dab.HostBuffer(n * 8)
        self.msc = dab.HostBuffer(n * g.P.nb_cifs * dab.CIF_OUT_STRIDE)

    def poison(self):
        for b in (self.log, self.index, self.status, self.msc):
            b.array[:] = 0xA5

    def kwargs(self, with_msc):
        kw = dict(dabplus=(self.log.ptr.value, self.log.nbytes, self.index.ptr.value), chan_status_host=self.status.ptr.value)
        if with_msc:
            kw["msc_host"] = self.msc.ptr.value
        return kw

    def index_view(self):
        return self.index.array.view(np.int32).reshape(self.n, self.g.max_subchannels, 2)


def twin_results(dab, g, first, n, n_subs):
    """what a context reports after its own decode: DAB+ logs + index through the getters, chan_status, MSC"""
    want = {(s, k): g.get_dabplus_events(s, k) for s in range(first, first + n) for k in range(n_subs)}
    _, index = raw_all(dab, g, first, n)
    status = [g.chan_status(s) for s in range(first, first + n)]
    msc = [[g.get_msc(s, k) for k in range(n_subs)] for s in range(first, first + n)]
    return want, index, status, msc


def check_ticket(dab, pyref, g, first, n, o, twin, with_msc, tag):
    want, index, status, msc = twin
    check_packed(dab, pyref, g, first, n, o.log.array, o.index_view(), want, tag)
    assert np.array_equal(o.index_view(), index), f"{tag}: index differs from the twin's"
    assert [tuple(r) for r in o.status.array.view(np.int32).reshape(n, 2)] == [tuple(x) for x in status], f"{tag}: chan_status"
    if with_msc:
        arena = o.msc.array.reshape(n, g.P.nb_cifs, -1)
        for c, per_sub in enumerate(msc):
            for k, (b, valid) in enumerate(per_sub):
                off, nb = g.msc_layout(first + c, k)
                for cif in np.nonzero(valid)[0]:
                    assert np.array_equal(arena[c, cif, off:off + nb], b[cif]), f"{tag}: stream {first + c} sub-channel {k}: MSC"


def test_pipelined_narrowband_equals_twin(gpu_ctx, tx, pyref):
    """dabgpu_submit_ex, two tickets in flight, 34 tickets of 0.3 - 1.4 frames, msc_host requested on two tickets of three; each
    ticket's DAB+ output equals a twin running ofdm_process + chan_decode + the per-sub getters; every input buffer is
    overwritten with noise as soon as its ticket was waited for"""
    dab = gpu_ctx
    S, FS = 3, tx.MODES[1].nb_frame_samples
    subs = tx.default_ensemble()[:3] + [tx.Subchannel(3, 144, 48, eep_level=2, dabplus=False), tx.Subchannel(4, 192, 12, eep_level=2)]
    iq = narrowband_iq(tx, subs, S, 34, seed=21)
    sizes = [int(FRACTIONS[i % 4] * FS) + 37 * (i % 3) for i in range(34)]
    assert 2 * sum(sizes) <= iq.shape[1]
    ga, gb = (dab.DabGpu(mode=1, max_streams=S, ring_samples=1 << 20) for _ in range(2))
    for g in (ga, gb):
        for s in range(S):
            g.msc_configure(s, subs)
    max_n = max(sizes)
    ins = [dab.HostBuffer(S * 2 * max_n, write_combined=True) for _ in range(2)]
    outs = [TicketOut(dab, gb, 0, S) for _ in range(2)]
    rng = np.random.default_rng(3)
    pending, pos = None, 0
    for i, m in enumerate(sizes):
        block = np.ascontiguousarray(iq[:, 2 * pos:2 * (pos + m)])
        pos += m
        ga.ofdm_process(block, block_size=BLOCK)
        ga.chan_decode()
        twin = twin_results(dab, ga, 0, S, len(subs))
        ins[i % 2].array.reshape(S, 2 * max_n)[:, :2 * m] = block
        outs[i % 2].poison()
        with_msc = i % 3 != 0
        t = gb.submit(ins[i % 2].ptr.value, 2 * max_n, m, block_size=BLOCK, run_chan_decode=True, **outs[i % 2].kwargs(with_msc))
        if pending is not None:
            tp, ip, wp, mp = pending
            gb.wait(tp)
            ins[ip % 2].array[:] = rng.integers(0, 256, ins[ip % 2].nbytes, dtype=np.uint8)
            check_ticket(dab, pyref, gb, 0, S, outs[ip % 2], wp, mp, f"ticket {ip}")
        pending = (t, i, twin, with_msc)
    tp, ip, wp, mp = pending
    gb.wait(tp)
    check_ticket(dab, pyref, gb, 0, S, outs[ip % 2], wp, mp, f"ticket {ip}")
    ca, cb = ga.counters(), gb.counters()
    assert ca == cb and ca["au_ok"] > 0 and ca["superframes_ok"] > 0
    ga.close()
    gb.close()


@pytest.mark.parametrize("name", ["k_wideband_s8", "k_wideband_mixed_s16"])
def test_pipelined_wideband_equals_twin(gpu_ctx, tx, pyref, name):
    """dabgpu_wideband_submit_ex against process + chan_decode + the getters on a twin, 30 tickets, two in flight; the mixed-rate
    configuration decodes a subset of the channels"""
    from test_wideband_pipeline_gpu import CONFIGS, Feed, open_front_end, ticket_sizes
    dab = gpu_ctx
    fs, fmt, _, offs, n_src, _ = CONFIGS[name]
    n_ch = n_src * len(offs)
    first, n = (1, n_ch - 3) if name == "k_wideband_mixed_s16" else (0, n_ch)
    ga, wa, _ = open_front_end(dab, tx, name)
    gb, wb, _ = open_front_end(dab, tx, name)
    sizes = ticket_sizes(tx, fs, 30)
    max_n = max(sizes)
    wb.reserve(max_n)
    feed = Feed(tx, name, seed=11)
    itemsize = feed.raw.itemsize
    ins = [dab.HostBuffer(n_src * max_n * 2 * itemsize, write_combined=True) for _ in range(2)]
    outs = [TicketOut(dab, gb, first, n) for _ in range(2)]
    rng = np.random.default_rng(12)
    pending = None
    for i, m in enumerate(sizes):
        block = feed.next(m)
        wa.process(block, block_size=BLOCK)
        ga.chan_decode(first, n)
        twin = twin_results(dab, ga, first, n, 4)
        ins[i % 2].array.view(block.dtype).reshape(n_src, max_n * 2)[:, :2 * m] = block
        outs[i % 2].poison()
        with_msc = i % 2 == 0
        t = wb.submit(ins[i % 2].ptr.value, max_n * 2 * itemsize, m, block_size=BLOCK, first_stream=first, n_streams=n,
                      run_chan_decode=True, **outs[i % 2].kwargs(with_msc))
        if pending is not None:
            tp, ip, wp, mp = pending
            gb.wait(tp)
            ins[ip % 2].array[:] = rng.integers(0, 256, ins[ip % 2].nbytes, dtype=np.uint8)
            check_ticket(dab, pyref, gb, first, n, outs[ip % 2], wp, mp, f"ticket {ip}")
        pending = (t, i, twin, with_msc)
    tp, ip, wp, mp = pending
    gb.wait(tp)
    check_ticket(dab, pyref, gb, first, n, outs[ip % 2], wp, mp, f"ticket {ip}")
    ca, cb = ga.counters(), gb.counters()
    assert ca == cb and ca["au_ok"] > 0
    for o in (wa, ga, wb, gb):
        o.close()


def test_full_size_1024_streams_18_subchannels(gpu_ctx, tx, pyref):
    """the benchmark's workload through dabgpu_submit_ex, two tickets in flight: every delivered AU is an AU of a superframe the
    transmitter sent on that stream's sub-channel, and the AU events equal the au_ok counter delta"""
    import torch
    dab = gpu_ctx
    synth = importlib.import_module(dab.__name__ + ".synth.gpusynth")
    S, PERIOD, WARM, CHECKED = 1024, 10, 10, 4
    subs = tx.default_ensemble()
    FS = tx.MODES[1].nb_frame_samples
    made = [tx.periodic_frames(1, subs, seed=4100 + u, period_frames=PERIOD, return_logical=True) for u in range(2)]
    sent = [[set() for _ in subs] for _ in made]   # AU payloads of every superframe sent, per unique ensemble and sub-channel
    for u, (_, logical) in enumerate(made):
        for k, sc in enumerate(subs):
            aac = pyref.PortAac()
            for fr in np.concatenate([logical[sc.id]] * 2):
                sent[u][k].update(e[5] for e in aac.process(fr) if e[0] == pyref.EV_AU)
            assert sent[u][k], (u, k)
    cyc, _, _ = synth.make_cyclic_streams_u8(S, np.stack([m[0] for m in made]), mode=1, seed0=77, snr_db=15.0, device="cuda:0")
    hb = dab.HostBuffer(S * 2 * PERIOD * FS)
    h_np = hb.array.reshape(S, 2 * PERIOD * FS)
    torch.from_numpy(h_np).copy_(cyc)
    del cyc
    torch.cuda.synchronize()
    g = dab.DabGpu(mode=1, max_streams=S)
    for s in range(S):
        g.msc_configure(s, subs)
    outs = [TicketOut(dab, g, 0, S) for _ in range(2)]
    n_au, c_start = 0, None

    def collect(j):
        nonlocal n_au
        got = dab.split_dabplus(outs[j % 2].log.array, outs[j % 2].index_view(), 0, g.max_subchannels)
        assert (outs[j % 2].status.array.view(np.int32).reshape(S, 2)[:, 0] == 1).all(), f"ticket {j}: a stream decoded no frame"
        for (s, k), v in got.items():
            for e in pyref.parse_event_log(v):
                assert e[0] in (pyref.EV_HEADER, pyref.EV_AU), f"ticket {j}: stream {s} sub-channel {k}: event {e[:5]}"
                if e[0] == pyref.EV_AU:
                    assert e[5] in sent[s % 2][k], f"ticket {j}: stream {s} sub-channel {k}: AU {e[1]} was not sent"
                    n_au += 1

    for phase, count in (("warm", WARM), ("checked", CHECKED)):
        pending = None
        for i in range(count):
            step = i if phase == "warm" else WARM + i
            view = h_np[:, 2 * (step % PERIOD) * FS:2 * ((step % PERIOD) + 1) * FS]
            outs[step % 2].poison()
            t = g.submit(view.ctypes.data, h_np.strides[0], FS, block_size=BLOCK, run_chan_decode=True, **outs[step % 2].kwargs(False))
            if pending is not None:
                g.wait(pending[0])
                if phase == "checked":
                    collect(pending[1])
            pending = (t, step)
        g.wait(pending[0])
        if phase == "checked":
            collect(pending[1])
        else:
            c_start = g.counters()
    d = {k: v - c_start[k] for k, v in g.counters().items()}
    assert d["au_ok"] == n_au and n_au >= S * len(subs) * 3 * CHECKED * 4 // 5 - S * len(subs) * 3
    assert d["superframes_rs_fail"] == 0 and d["superframes_firecode_fail"] == 0 and d["au_crc_fail"] == 0
    g.close()
    hb.close()


def test_refusals_leave_the_context_unchanged(gpu_ctx, tx, pyref):
    """context A tries log_cap one byte below the bound, a NULL index and DAB+ output without a channel decode before each valid
    dabgpu_submit_ex; B runs dabgpu_submit and the synchronous batch getter; C runs dabgpu_submit_ex with dabplus = NULL.  All
    three report the same, and A's DAB+ output is B's."""
    dab = gpu_ctx
    S, FS = 2, tx.MODES[1].nb_frame_samples
    subs = tx.default_ensemble()[:2] + [tx.Subchannel(2, 96, 48, eep_level=2, dabplus=False)]
    iq = narrowband_iq(tx, subs, S, 12, seed=41)
    ctxs = [dab.DabGpu(mode=1, max_streams=S) for _ in range(3)]
    for g in ctxs:
        for s in range(S):
            g.msc_configure(s, subs)
    A, B, Cc = ctxs
    ins = dab.HostBuffer(S * 2 * FS)
    outs = [TicketOut(dab, g, 0, S) for g in ctxs]
    bound = A.dabplus_out_bound(0, S)
    assert bound > 0 and bound == B.dabplus_out_bound(0, S)
    n_events = 0
    for i in range(11):
        ins.array.reshape(S, 2 * FS)[:] = iq[:, 2 * i * FS:2 * (i + 1) * FS]
        for o in outs:
            o.poison()
        p, stride = ins.ptr.value, 2 * FS
        o = outs[0]
        launches = A.launch_count
        for dp, run, code in (((o.log.ptr.value, bound - 1, o.index.ptr.value), True, dab.ERR_OVERFLOW),
                              ((o.log.ptr.value, bound, None), True, dab.ERR_INVALID),
                              ((o.log.ptr.value, bound, o.index.ptr.value), False, dab.ERR_INVALID)):
            with pytest.raises(dab.DabGpuError) as e:
                A.submit(p, stride, FS, block_size=BLOCK, run_chan_decode=run, dabplus=dp, chan_status_host=o.status.ptr.value)
            assert e.value.code == code, (i, dp, run, str(e.value))
        assert A.launch_count == launches
        A.wait(A.submit(p, stride, FS, block_size=BLOCK, run_chan_decode=True, **o.kwargs(True)))
        B.wait(B.submit(p, stride, FS, block_size=BLOCK, run_chan_decode=True, chan_status_host=outs[1].status.ptr.value,
                        msc_host=outs[1].msc.ptr.value))
        st = dab._step(p, stride, FS, BLOCK, 0, S, True, {"chan_status_host": outs[2].status.ptr.value, "msc_host": outs[2].msc.ptr.value})
        t = C.c_uint64(0)
        dab._check(Cc.L.dabgpu_submit_ex(Cc.h, C.byref(st), None, C.byref(t)))
        Cc.wait(t.value)
        for other in outs[1:]:
            assert np.array_equal(o.status.array, other.status.array) and np.array_equal(o.msc.array, other.msc.array), f"ticket {i}"
        log_b, index_b = raw_all(dab, B, 0, S)
        want = dab.split_dabplus(log_b, index_b, 0, B.max_subchannels)
        assert np.array_equal(o.index_view(), index_b), f"ticket {i}: index"
        got = check_packed(dab, pyref, A, 0, S, o.log.array, o.index_view(), want, f"ticket {i}")
        n_events += len(got)
    assert n_events > 0 and A.counters() == B.counters() == Cc.counters()
    for g in ctxs:
        g.close()
