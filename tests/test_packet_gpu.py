"""Packet-mode sub-channels in the channel decode on the GPU (k_packet, k_packet_pack).

Oracle everywhere: tests/packet_cases.py's processor (PortPacketFec plus the packet records) fed the GPU's own
dabgpu_chan_get_msc bytes of the same decode, entry by entry; every log must equal it byte for byte, through the per-sub
getter, the packed getter and the pipelined tickets."""
import ctypes as C
import dataclasses

import numpy as np
import pytest

import packet_cases as pc
from test_dabplus_out_gpu import BLOCK, TicketOut, check_packed, narrowband_iq, raw_all, twin_results

pytestmark = pytest.mark.gpu


def mixed_subs(tx):
    """DAB+, STREAM and packet entries with and without FEC: EEP-A and -B, one UEP row, 8 to 384 kbit/s"""
    return [tx.Subchannel(0, 0, 48, eep_level=2),
            tx.Subchannel(1, 48, 48, eep_level=2, dabplus=False),
            tx.Subchannel(2, 96, 12, eep_level=0, packet_fec=True),                       # 8 kbit/s 1-A
            tx.Subchannel(3, 108, 18, eep_level=2, eep_type_b=True, packet_fec=True),     # 32 kbit/s 3-B
            tx.Subchannel(4, 126, 32, is_uep=True, uep_index=14, packet_fec=False),       # UEP row 14, 64 kbit/s
            tx.Subchannel(5, 158, 192, eep_level=3, packet_fec=True),                     # 384 kbit/s 4-A
            tx.Subchannel(6, 350, 24, eep_level=1, packet_fec=False)]                     # 24 kbit/s 2-A


def as_stream(subs):
    return [dataclasses.replace(sc, packet_fec=None, dabplus=False) if sc.packet_fec is not None else sc for sc in subs]


class Oracles:
    """one oracle processor per (stream, packet entry), fed what the GPU decoded"""

    def __init__(self, pyref, tx, stream_subs):
        self.pyref, self.tx = pyref, tx
        self.o = {}
        self.logs = {}            # (s, k) -> every record of the run
        for s, subs in enumerate(stream_subs):
            for k, sc in enumerate(subs):
                if sc.packet_fec is not None:
                    self.attach(s, k, sc.packet_fec)

    def attach(self, s, k, fec):
        self.o[(s, k)] = pc.make_oracle(self.pyref, self.tx, fec)
        self.logs.setdefault((s, k), b"")

    def detach(self, s, k):
        self.o.pop((s, k), None)

    def decoded(self, g, streams, tag):
        """after a chan_decode of `streams`: each entry's per-sub getter equals its oracle; returns {(s, k): log}"""
        want = {}
        for (s, k), o in self.o.items():
            if s not in streams:
                continue
            exp = b""
            if g.chan_status(s)[0]:
                out, valid = g.get_msc(s, k)
                for c in range(g.P.nb_cifs):
                    if valid[c]:
                        exp += o.frame(out[c])
            got = g.get_dabplus_events(s, k)
            assert got == exp, f"{tag}: stream {s} entry {k}: {pc.parse(got)[:3]} != {pc.parse(exp)[:3]}"
            self.logs[(s, k)] += exp
            want[(s, k)] = exp
        return want


def delivered(log):
    return [(e[5], e[1], e[2]) for e in pc.parse(log) if e[0] == pc.EV_PACKET]


def run(dab, tx, pyref, mode, stream_subs, n_frames, hooks=None, snr_db=None, twin=False):
    S = len(stream_subs)
    enss = [tx.EnsembleTx(mode, stream_subs[s], seed=40 + 9 * s, packet_hook=(hooks or [None] * S)[s]) for s in range(S)]
    g = dab.DabGpu(mode=mode, max_streams=S)
    gt = dab.DabGpu(mode=mode, max_streams=S) if twin else None
    for s in range(S):
        g.msc_configure(s, stream_subs[s])
        if gt:
            gt.msc_configure(s, as_stream(stream_subs[s]))
    ref = Oracles(pyref, tx, stream_subs)
    rng = np.random.default_rng(mode)
    for f in range(n_frames):
        soft = np.stack([tx.hard_to_soft(e.next_frame_bits(), rng, (snr_db or [None] * S)[s]) for s, e in enumerate(enss)])
        for x in (g, gt) if gt else (g,):
            x.softbits_push(soft)
            x.chan_decode()
        want = ref.decoded(g, range(S), f"mode {mode} frame {f}")
        got = g.get_dabplus_all()
        for key, v in want.items():
            assert got.get(key, b"") == v, f"frame {f}: packed {key}"
        for (s, k), v in got.items():
            if (s, k) not in want:
                assert v == g.get_dabplus_events(s, k)
        if gt:   # the packet entries change nothing else: MSC bytes, FIBs, DAB+ logs
            for s in range(S):
                assert g.chan_status(s) == gt.chan_status(s)
                fa, fb = g.get_fic(s), gt.get_fic(s)
                assert np.array_equal(fa[0], fb[0]) and np.array_equal(fa[1], fb[1])
                for k, sc in enumerate(stream_subs[s]):
                    ma, mb = g.get_msc(s, k), gt.get_msc(s, k)
                    assert np.array_equal(ma[0], mb[0]) and np.array_equal(ma[1], mb[1])
                    if sc.packet_fec is None:
                        assert g.get_dabplus_events(s, k) == gt.get_dabplus_events(s, k)
    if gt:
        assert g.counters() == gt.counters()
        gt.close()
    g.close()
    return enss, ref


@pytest.mark.parametrize("mode", [1, 2, 4])
def test_mixed_table_clean(gpu_ctx, tx, pyref, mode):
    """every delivered packet is a transmitted one, in order, with is_corrected = crc_ok = 1 (with FEC) or crc_ok = 1 (without)"""
    subs = mixed_subs(tx)
    n_frames = {1: 40, 2: 150, 4: 80}[mode]
    enss, ref = run(gpu_ctx, tx, pyref, mode, [subs, subs], n_frames)
    for (s, k), log in ref.logs.items():
        sc = subs[k]
        sent = [p.tobytes() for p in enss[s].packets[sc.id] if not (sc.packet_fec and pc.address(p.tobytes()) == pc.FEC_ADDRESS)]
        got = delivered(log)
        assert len(got) > 0 and [p for p, _, _ in got] == sent[:len(got)], (s, k)
        assert all(ok == 1 and (c == 1) == bool(sc.packet_fec) for _, c, ok in got), (s, k)
        fec = [e for e in pc.parse(log) if e[0] == pc.EV_PACKET_FEC]
        if sc.packet_fec and sc.frame_bytes >= 96:
            assert fec and all(e[1:5] == (1, 12, 0, 0) for e in fec), (s, k)


def test_scenarios_with_channel_noise_and_twin(gpu_ctx, tx, pyref):
    """every scenario of make_packet_fec_golden through the transmitter hook, Viterbi output with errors from channel noise;
    a twin context with the packet entries declared STREAM reports the same MSC bytes, FIBs, DAB+ logs and counters"""
    subs = mixed_subs(tx)
    hooks = [pc.scenario_hook(tx, 1), pc.scenario_hook(tx, 2)]
    _, ref = run(gpu_ctx, tx, pyref, 1, [subs, subs], 60, hooks=hooks, snr_db=[6.0, 1.0], twin=True)
    fec = [e for log in ref.logs.values() for e in pc.parse(log) if e[0] == pc.EV_PACKET_FEC]
    pk = [e for log in ref.logs.values() for e in pc.parse(log) if e[0] == pc.EV_PACKET]
    assert any(e[1] == 1 for e in fec) and any(e[1] == 0 for e in fec)
    assert any(e[2] == 0 for e in pk) and any(e[2] == 1 for e in pk)


def adversarial_frames(tx, sc, phase):
    """all 24-byte packets: 4 logical frames of data packets (they fill the ring), then 4 of FEC packets whose counter is broken
    (each ends a set: the first releases the whole ring, every one releases itself)"""
    rng = np.random.default_rng(phase)
    nb, count = sc.frame_bytes, [0]

    def frame(_sc):
        i = count[0]
        count[0] += 1
        if (i + phase) % 8 < 4:
            return np.concatenate([tx.data_packet(rng, 24, 7, j & 3, True, True) for j in range(nb // 24)])
        p = rng.integers(0, 256, size=(nb // 24, 24), dtype=np.uint8)
        p[:, 0], p[:, 1] = (5 << 2) | 0x03, 0xFE
        return p.reshape(-1)

    return frame


def test_packed_bound_overflow_and_adversarial_stream(gpu_ctx, tx, pyref):
    dab = gpu_ctx
    sc = tx.Subchannel(0, 0, 192, eep_level=2, packet_fec=True)      # 256 kbit/s, 768 bytes per logical frame
    subs = [sc, tx.Subchannel(1, 192, 48, eep_level=2)]
    S = 4
    enss = [tx.EnsembleTx(1, subs, seed=s) for s in range(S)]
    for s, e in enumerate(enss):
        fresh, adv = e._next_logical_frame, adversarial_frames(tx, sc, s)
        e._next_logical_frame = lambda x, fresh=fresh, adv=adv: adv(x) if x.id == 0 else fresh(x)
    g = dab.DabGpu(mode=1, max_streams=S)
    for s in range(S):
        g.msc_configure(s, subs)
    ref = Oracles(pyref, tx, [subs] * S)
    A = 4 * sc.frame_bytes
    bound_item = 24 * ((2472 + A) // 24) + 2472 + A + 24 * (A // 24 + 1)
    dp_one = g.dabplus_out_bound(0, 1)
    assert dp_one >= bound_item
    peak = 0
    for f in range(30):
        g.softbits_push(np.stack([tx.hard_to_soft(e.next_frame_bits()) for e in enss]))
        g.chan_decode()
        want = ref.decoded(g, range(S), f"frame {f}")
        peak = max([peak] + [len(v) for v in want.values()])
        assert all(len(v) <= bound_item for v in want.values())
        log, index = raw_all(dab, g, 0, S)
        dp_want = {(s, 1): g.get_dabplus_events(s, 1) for s in range(S)}
        dp_want.update(want)
        check_packed(dab, pyref, g, 0, S, log, index, dp_want, f"frame {f}")
        if f == 20:   # a cap below the bound is refused before anything is queued
            bound = g.dabplus_out_bound(0, S)
            small = np.zeros(bound - 1, dtype=np.uint8)
            idx = np.zeros((S, g.max_subchannels, 2), dtype=np.int32)
            out = dab.DabPlusOut(small.ctypes.data, small.size, idx.ctypes.data)
            assert g.L.dabgpu_chan_get_dabplus_all(g.h, 0, S, C.byref(out)) == dab.ERR_OVERFLOW
    assert peak >= 0.95 * bound_item, (peak, bound_item)
    g.close()


def test_invalid_payloads(gpu_ctx, tx):
    dab = gpu_ctx
    g = dab.DabGpu(mode=1, max_streams=1)
    e = dab.SubchannelExC()
    dab.DabGpu._fill_sub(e, tx.Subchannel(0, 0, 12, eep_level=0, packet_fec=True))
    e.sc.is_dabplus = 1
    idx = C.c_int(-1)
    assert g.L.dabgpu_msc_add_subchannel_ex(g.h, 0, C.byref(e), C.byref(idx)) == dab.ERR_INVALID
    e.sc.is_dabplus, e.payload = 0, 9
    assert g.L.dabgpu_msc_configure_ex(g.h, 0, C.byref(e), 1) == dab.ERR_INVALID
    g.close()


def test_table_changes_between_decodes(gpu_ctx, tx, pyref):
    """add, remove, configure_ex and a kind change between decodes; an unchanged entry keeps a set that spans the change"""
    dab = gpu_ctx
    subs = mixed_subs(tx)
    ens = tx.EnsembleTx(1, subs, seed=8)
    g = dab.DabGpu(mode=1, max_streams=1)
    table = subs[:4]
    g.msc_configure(0, table)
    ref = Oracles(pyref, tx, [table])
    for f in range(36):
        if f == 8:        # add the 384 kbit/s FEC entry and the UEP packet entry
            for sc in (subs[5], subs[4]):
                k = g.msc_add_subchannel(0, sc)
                ref.attach(0, k, sc.packet_fec)
        if f == 14:       # remove the 32 kbit/s FEC entry
            g.msc_remove_subchannel(0, 3)
            ref.detach(0, 3)
        if f == 20:       # the same table again with entry 2 unchanged (its 8 kbit/s set spans the change), entry 4 turned into STREAM,
            #              entry 3 back, and entry 5 changed from FEC to plain packets
            t2 = [subs[0], subs[1], subs[2], subs[3]] + as_stream([subs[5], subs[4]])
            keep = ref.o[(0, 2)]
            g.msc_configure(0, t2)
            ref.o = {(0, 2): keep}
            ref.attach(0, 3, True)
        if f == 28:       # kind change of entry 4 (stream -> packets without FEC), entry 5 stream -> FEC
            t3 = [subs[0], subs[1], subs[2], subs[3], dataclasses.replace(subs[5], packet_fec=False), subs[4]]
            keep = {key: ref.o[key] for key in ((0, 2), (0, 3))}
            g.msc_configure(0, t3)
            ref.o = keep
            ref.attach(0, 4, False)
            ref.attach(0, 5, False)
        g.softbits_push(tx.hard_to_soft(ens.next_frame_bits())[None])
        g.chan_decode()
        want = ref.decoded(g, [0], f"frame {f}")
        got = g.get_dabplus_all()
        for key, v in want.items():
            assert got.get(key, b"") == v
    # the 8 kbit/s entry was never reset: its packets are the transmitted ones, corrected, in order
    sent = [p.tobytes() for p in ens.packets[2] if pc.address(p.tobytes()) != pc.FEC_ADDRESS]
    got = delivered(ref.logs[(0, 2)])
    assert len(got) > 0 and [p for p, _, _ in got] == sent[:len(got)] and all(c == 1 for _, c, _ in got)
    g.close()


def test_pipelined_submit_equals_twin(gpu_ctx, tx, pyref):
    """dabgpu_submit_ex with two tickets in flight: the packed logs of the packet entries equal a twin's process + chan_decode +
    getters"""
    dab = gpu_ctx
    S, FS = 2, tx.MODES[1].nb_frame_samples
    subs = mixed_subs(tx)
    iq = narrowband_iq(tx, subs, S, 16, seed=5)
    sizes = [int((0.3, 1.0, 0.7, 1.4)[i % 4] * FS) for i in range(14)]
    ga, gb = (dab.DabGpu(mode=1, max_streams=S, ring_samples=1 << 20) for _ in range(2))
    for g in (ga, gb):
        for s in range(S):
            g.msc_configure(s, subs)
    max_n = max(sizes)
    ins = [dab.HostBuffer(S * 2 * max_n, write_combined=True) for _ in range(2)]
    outs = [TicketOut(dab, gb, 0, S) for _ in range(2)]
    pending, pos, n_packets = None, 0, 0
    for i, m in enumerate(sizes):
        block = np.ascontiguousarray(iq[:, 2 * pos:2 * (pos + m)])
        pos += m
        ga.ofdm_process(block, block_size=BLOCK)
        ga.chan_decode()
        want, index, _, _ = twin_results(dab, ga, 0, S, len(subs))
        n_packets += sum(len(delivered(want[(s, k)])) for s in range(S) for k in (2, 3, 4, 5, 6))
        ins[i % 2].array.reshape(S, 2 * max_n)[:, :2 * m] = block
        outs[i % 2].poison()
        t = gb.submit(ins[i % 2].ptr.value, 2 * max_n, m, block_size=BLOCK, run_chan_decode=True, **outs[i % 2].kwargs(False))
        if pending is not None:
            tp, ip, wp, xp = pending
            gb.wait(tp)
            check_packed(dab, pyref, gb, 0, S, outs[ip % 2].log.array, outs[ip % 2].index_view(), wp, f"ticket {ip}")
            assert np.array_equal(outs[ip % 2].index_view(), xp)
        pending = (t, i, want, index)
    tp, ip, wp, xp = pending
    gb.wait(tp)
    check_packed(dab, pyref, gb, 0, S, outs[ip % 2].log.array, outs[ip % 2].index_view(), wp, f"ticket {ip}")
    assert n_packets > 0 and ga.counters() == gb.counters()


def test_ring_overrun_skip_continues_with_decoded_frames(gpu_ctx, tx, pyref):
    """the OFDM stage runs seven frames ahead of the channel decoder, further than the 8-slot frame ring keeps history: the decoder
    skips to the newest frame (chan_pick_frame) and restarts its time de-interleavers, while the packet entries' FEC rings are not
    touched and simply continue with the frames that are decoded; the oracle stays "the processor fed the emitted frames"."""
    dab = gpu_ctx
    subs = mixed_subs(tx)
    ens = tx.EnsembleTx(1, subs, seed=17)
    n_frames, block = 64, 65536
    iq = tx.ofdm_modulate([ens.next_frame_bits() for _ in range(n_frames)], 1)
    u8 = tx.to_u8(tx.impair(iq, 20.0, 0.4e-3, 999, seed=2, tail_samples=3000), 30.0)
    g = dab.DabGpu(mode=1, max_streams=1, frame_slots=8)
    g.msc_configure(0, subs)
    ref = Oracles(pyref, tx, [subs])
    n = (u8.size // 2 // block) * block
    held, fill_at_skip = range(60 * block, 81 * block), None
    for off in range(0, n, block):
        g.ofdm_process(u8[None, 2 * off:2 * (off + block)], block_size=block)
        if off in held:
            continue                                   # the decoder stalls: about seven frames pile up in the ring
        if fill_at_skip is None and off == held.stop:
            fill_at_skip = (ref.o[(0, 2)].fill, ref.o[(0, 3)].fill)
        while True:
            d0 = g.counters()["frames_dropped"]
            g.chan_decode()
            if not g.chan_status(0)[0]:
                break
            ref.decoded(g, [0], f"block {off // block}")
            if g.counters()["frames_dropped"] > d0:
                assert off == held.stop
    assert g.counters()["frames_dropped"] > 0
    assert fill_at_skip[0] > 0 and fill_at_skip[1] > 0     # FEC sets in progress across the skip
    for k in (2, 3, 5):
        fec = [e for e in pc.parse(ref.logs[(0, k)]) if e[0] == pc.EV_PACKET_FEC]
        assert fec, k
    g.close()


@pytest.mark.parametrize("name", ["k_wideband_s8", "k_wideband_mixed_s16"])
def test_pipelined_wideband_equals_twin(gpu_ctx, tx, pyref, name):
    """dabgpu_wideband_submit_ex with packet entries (with and without FEC) next to DAB+ ones, two tickets in flight: each ticket's
    packed logs and index equal a twin's process + chan_decode + getters, and the twin's packet logs equal the oracle fed its MSC
    bytes.  The front end's ensembles carry DAB+ superframes on every sub-channel, so the packet entries cut them as packets."""
    from test_dabplus_out_gpu import check_ticket
    from test_wideband_pipeline_gpu import CONFIGS, Feed, open_front_end, ticket_sizes
    dab = gpu_ctx
    fs, fmt, _, offs, n_src, _ = CONFIGS[name]
    n_ch = n_src * len(offs)
    first, n = (1, n_ch - 3) if name == "k_wideband_mixed_s16" else (0, n_ch)
    base = tx.default_ensemble()[:4]
    table = base[:2] + [dataclasses.replace(base[2], packet_fec=True), dataclasses.replace(base[3], packet_fec=False)]
    ga, wa, _ = open_front_end(dab, tx, name)
    gb, wb, _ = open_front_end(dab, tx, name)
    for g in (ga, gb):
        for c in range(n_ch):
            g.msc_configure(c, table)
    ref = Oracles(pyref, tx, [table] * n_ch)
    sizes = ticket_sizes(tx, fs, 24)
    max_n = max(sizes)
    wb.reserve(max_n)
    feed = Feed(tx, name, seed=11)
    itemsize = feed.raw.itemsize
    ins = [dab.HostBuffer(n_src * max_n * 2 * itemsize, write_combined=True) for _ in range(2)]
    outs = [TicketOut(dab, gb, first, n) for _ in range(2)]
    pending = None
    for i, m in enumerate(sizes):
        block = feed.next(m)
        wa.process(block, block_size=BLOCK)
        ga.chan_decode(first, n)
        ref.decoded(ga, range(first, first + n), f"ticket {i}")
        twin = twin_results(dab, ga, first, n, 4)
        ins[i % 2].array.view(block.dtype).reshape(n_src, max_n * 2)[:, :2 * m] = block
        outs[i % 2].poison()
        t = wb.submit(ins[i % 2].ptr.value, max_n * 2 * itemsize, m, block_size=BLOCK, first_stream=first, n_streams=n,
                      run_chan_decode=True, **outs[i % 2].kwargs(False))
        if pending is not None:
            tp, ip, wp = pending
            gb.wait(tp)
            check_ticket(dab, pyref, gb, first, n, outs[ip % 2], wp, False, f"ticket {ip}")
        pending = (t, i, twin)
    tp, ip, wp = pending
    gb.wait(tp)
    check_ticket(dab, pyref, gb, first, n, outs[ip % 2], wp, False, f"ticket {ip}")
    assert sum(len(delivered(v)) for v in ref.logs.values()) > 0
    assert ga.counters() == gb.counters()
    for o in (wa, ga, wb, gb):
        o.close()


def _sent_index(tx, subs, logical, k):
    """{packet bytes: position} of the data packets a sub-channel sends in one period (its logical frames cut into packets); padding
    packets (address 0) are all alike and get no position"""
    out, pos = {}, 0
    for fr in logical[subs[k].id]:
        off = 0
        while off < fr.size:
            n = 24 * ((int(fr[off]) >> 6) + 1)
            p = fr[off:off + n].tobytes()
            if pc.address(p) not in (0, pc.FEC_ADDRESS):
                out[p] = pos
                pos += 1
            off += n
    return out, pos


def _full_size_run(dab, tx, synth, subs, made, S, PERIOD, WARM, CHECKED, check):
    import torch
    FS = tx.MODES[1].nb_frame_samples
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
    c_start = None
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
                    check(g, outs[pending[1] % 2], pending[1])
            pending = (t, step)
        g.wait(pending[0])
        if phase == "checked":
            check(g, outs[pending[1] % 2], pending[1])
        else:
            c_start = g.counters()
    d = {k: v - c_start[k] for k, v in g.counters().items()}
    g.close()
    hb.close()
    return d


def test_full_size_1024_streams_16_dabplus_2_packet_fec(gpu_ctx, tx, pyref):
    """the benchmark's workload with two of the 18 sub-channels of every stream carrying FEC-protected packets, through OFDM and
    dabgpu_submit_ex, two tickets in flight: every crc_ok packet is a data packet that stream's sub-channel sent, in sending
    order (cyclically: the payload repeats every PERIOD frames), and the counter deltas equal those of the same run with the two
    entries declared STREAM.  The packet stream wraps at the period seam, so a set that crosses it is abandoned or fails rows:
    only crc_ok packets are counted."""
    import importlib
    dab = gpu_ctx
    synth = importlib.import_module(dab.__name__ + ".synth.gpusynth")
    S, PERIOD, WARM, CHECKED = 1024, 10, 10, 6
    subs = [dataclasses.replace(sc, packet_fec=True) if sc.id >= 16 else sc for sc in tx.default_ensemble()]
    made = [tx.periodic_frames(1, subs, seed=4200 + u, period_frames=PERIOD, return_logical=True) for u in range(2)]
    sent = [{k: _sent_index(tx, subs, logical, k) for k in (16, 17)} for _, logical in made]
    last, n_ok = {}, [0]

    def check(g, o, j):
        st = o.status.array.view(np.int32).reshape(S, 2)
        assert (st[:, 0] == 1).all(), f"ticket {j}: a stream decoded no frame"
        got = dab.split_dabplus(o.log.array, o.index_view(), 0, g.max_subchannels)
        for (s, k), v in got.items():
            if k < 16:
                continue
            index, n_sent = sent[s % 2][k]
            for e in pc.parse(v):
                if e[0] != pc.EV_PACKET or not e[2] or e[3] == 0:
                    continue
                assert e[5] in index, f"ticket {j}: stream {s} entry {k}: a crc_ok packet that was not sent"
                p = index[e[5]]
                if (s, k) in last:
                    step = (p - last[(s, k)]) % n_sent
                    assert 0 < step <= n_sent // 2, f"ticket {j}: stream {s} entry {k}: packet {p} after {last[(s, k)]}"
                last[(s, k)] = p
                n_ok[0] += 1

    d = _full_size_run(dab, tx, synth, subs, made, S, PERIOD, WARM, CHECKED, check)
    assert n_ok[0] >= S * 2 * CHECKED * 4, n_ok[0]        # 8 packets of a 192-byte frame, 4 frames per ticket, most sets decoded
    assert len(last) == 2 * S
    d_stream = _full_size_run(dab, tx, synth, as_stream(subs), made, S, PERIOD, WARM, CHECKED, lambda g, o, j: None)
    assert d == d_stream and d["au_ok"] > 0
