"""Pipelined wideband front end (dabgpu_wideband_reserve / _submit, tickets retired with dabgpu_wait) on the GPU: every ticket's
copied results equal those of dabgpu_wideband_process + dabgpu_chan_decode + the getters on a twin context, whatever the ticket
sizes, with the input buffer overwritten as soon as its ticket is waited for, mixed with process calls and closed with tickets
in flight; the ring size does not change the output; a full-size round trip through submit alone; argument validation."""
import numpy as np
import pytest

from test_wideband_gpu import PERIOD, WARM, _hash
from test_wideband_gpu import make_capture as make_capture_pow2
from test_wideband_rates_gpu import make_capture as make_capture_any

pytestmark = pytest.mark.gpu

CAP = 1 << 19
BLOCK = 65536
FRACTIONS = (0.3, 1.0, 0.7, 1.4)   # ticket sizes in frames of input; most are not multiples of step_in
# (rate, format, quantiser rms, offsets, sources, any_rate): k_wideband at 8.192 MHz and k_wideband_mixed at 10 MS/s
CONFIGS = {
    "k_wideband_s8": (8192000, "raw_s8", 40.0, [-2568000, -856000, 856000, 2568000], 4, False),
    "k_wideband_mixed_s16": (10000000, "raw_s16l", 3000.0, [-1712000, 0, 1712000], 3, True),
}
OUT_FIELDS = ("frames", "produced", "msc", "msc_valid", "fic", "fic_crc", "chan_status")


def frame_input(tx, fs):
    return tx.MODES[1].nb_frame_samples * fs // 2048000


def ticket_sizes(tx, fs, n):
    step = frame_input(tx, fs)
    return [int(FRACTIONS[i % len(FRACTIONS)] * step) + 37 * (i % 3) for i in range(n)]


class Feed:
    """The raw input of every source of one configuration, cut into consecutive calls."""

    def __init__(self, tx, name, seed):
        fs, fmt, rms, offs, n_src, _ = CONFIGS[name]
        if fs % 2048000 == 0:
            cap, _ = make_capture_pow2(tx, fs // 2048000, offs, [61 + k for k in range(len(offs))], seed=seed)
        else:
            cap, _ = make_capture_any(tx, fs, offs, [61 + k for k in range(len(offs))], seed=seed)
        self.raw = tx.quantize(cap, fmt, rms).reshape(-1, 2)
        self.leads = [(s * 7919 * 37) % self.raw.shape[0] for s in range(n_src)]
        self.pos = 0

    def next(self, n):
        out = np.stack([np.take(self.raw, np.arange(ld + self.pos, ld + self.pos + n), axis=0, mode="wrap").reshape(-1)
                        for ld in self.leads])
        self.pos += n
        return out


def open_front_end(dab, tx, name):
    import torch
    fs, fmt, _, offs, n_src, any_rate = CONFIGS[name]
    channels = [(s, f) for s in range(n_src) for f in offs]
    g = dab.DabGpu(mode=1, max_streams=len(channels), iq_format=dab.IQ_C32)
    out = torch.zeros((len(channels), CAP), dtype=torch.complex64, device="cuda:0")
    w = g.wideband_open(fs, fmt, [c[0] for c in channels], [c[1] for c in channels], out.data_ptr(), CAP, any_rate=any_rate)
    for c in range(len(channels)):
        g.msc_configure(c, tx.default_ensemble()[:4])
    return g, w, out


class Outputs:
    """Pinned result buffers of one ticket, in dabgpu_step's layouts for n channels."""

    def __init__(self, dab, P, n):
        nc = P.nb_cifs
        sizes = dict(frames=n * P.nb_frame_bits, produced=n, msc=n * nc * dab.CIF_OUT_STRIDE, msc_valid=n * nc * 64,
                     fic=n * nc * dab.FIC_GROUP_STRIDE, fic_crc=n * nc * 4, chan_status=n * 8)
        self.n, self.P = n, P
        self.bufs = {k: dab.HostBuffer(sizes[k]) for k in OUT_FIELDS}

    def ptrs(self):
        return {k + "_host": self.bufs[k].ptr.value for k in OUT_FIELDS}

    def poison(self):
        for b in self.bufs.values():
            b.array[:] = 0xA5

    def view(self):
        n, nc = self.n, self.P.nb_cifs
        a = {k: self.bufs[k].array for k in OUT_FIELDS}
        return dict(frames=a["frames"].view(np.int8).reshape(n, -1), produced=a["produced"],
                    msc=a["msc"].reshape(n, nc, -1), msc_valid=a["msc_valid"].reshape(n, nc, 64),
                    fic=a["fic"].reshape(n, nc, -1), fic_crc=a["fic_crc"].reshape(n, nc, 4),
                    chan_status=a["chan_status"].view(np.int32).reshape(n, 2))


def serial_results(g, first, n, n_subs, pop=True):
    """what the getters report after process + chan_decode(first, n): per channel (status, fic, crc, [(msc, valid)], popped)"""
    res = []
    for ch in range(first, first + n):
        fibs, ok = g.get_fic(ch)
        popped = g.ofdm_pop_frames(ch, max_frames=8) if pop else None
        res.append((g.chan_status(ch), fibs, ok, [g.get_msc(ch, k) for k in range(n_subs)], popped))
    return res


def check_ticket(tag, g, first, got, want, frames=True):
    P = g.P
    nf, nc = P.nb_fibs_per_cif, P.nb_cifs
    for c, (status, fibs, ok, msc, popped) in enumerate(want):
        ch = first + c
        assert tuple(got["chan_status"][c]) == tuple(status), f"{tag}: channel {ch}: chan_status"
        assert np.array_equal(got["fic"][c, :, :nf * 32].reshape(nc * nf, 32), fibs), f"{tag}: channel {ch}: FIBs"
        assert np.array_equal(got["fic_crc"][c, :, :nf].reshape(-1), ok), f"{tag}: channel {ch}: FIB CRC flags"
        for k, (bytes_k, valid_k) in enumerate(msc):
            off, nb = g.msc_layout(ch, k)
            assert np.array_equal(got["msc"][c, :, off:off + nb], bytes_k), f"{tag}: channel {ch} sub-channel {k}: MSC bytes"
            assert np.array_equal(got["msc_valid"][c, :, k], valid_k), f"{tag}: channel {ch} sub-channel {k}: MSC valid flags"
        if frames:
            assert got["produced"][c] == (len(popped) > 0), f"{tag}: channel {ch}: produced flag"
            if popped:
                assert np.array_equal(got["frames"][c], popped[-1][0]), f"{tag}: channel {ch}: newest frame"


@pytest.mark.parametrize("name", list(CONFIGS))
@pytest.mark.parametrize("subset", [False, True], ids=["all-channels", "subset"])
def test_tickets_equal_process_and_chan_decode(gpu_ctx, tx, name, subset):
    """two tickets in flight (wait for t - 1 after submitting t), 44 tickets of 0.3 / 1.0 / 0.7 / 1.4 frames so the input ring
    wraps several times, every output pointer; the input buffer of a ticket is overwritten with noise as soon as it is waited
    for"""
    dab = gpu_ctx
    fs, fmt, _, offs, n_src, _ = CONFIGS[name]
    n_ch = n_src * len(offs)
    first, n = (1, n_ch - 3) if subset else (0, n_ch)
    n_subs = 4
    ga, wa, _ = open_front_end(dab, tx, name)
    gb, wb, _ = open_front_end(dab, tx, name)
    sizes = ticket_sizes(tx, fs, 44)
    max_n = max(sizes)
    wb.reserve(max_n)
    feed = Feed(tx, name, seed=5)
    itemsize = feed.raw.itemsize
    ins = [dab.HostBuffer(n_src * max_n * 2 * itemsize, write_combined=True) for _ in range(2)]
    outs = [Outputs(dab, gb.P, n) for _ in range(2)]
    rng = np.random.default_rng(9)
    pending = None   # (ticket, index, expected results)
    for i, m in enumerate(sizes):
        block = feed.next(m)
        wa.process(block, block_size=BLOCK)
        ga.chan_decode(first, n)
        want = serial_results(ga, first, n, n_subs)
        buf = ins[i % 2].array.view(block.dtype).reshape(n_src, max_n * 2)
        buf[:, :2 * m] = block
        outs[i % 2].poison()
        t = wb.submit(ins[i % 2].ptr.value, max_n * 2 * itemsize, m, block_size=BLOCK, first_stream=first, n_streams=n,
                      run_chan_decode=True, **outs[i % 2].ptrs())
        if pending is not None:
            tp, ip, wp = pending
            gb.wait(tp)
            ins[ip % 2].array[:] = rng.integers(0, 256, ins[ip % 2].nbytes, dtype=np.uint8)
            check_ticket(f"ticket {ip}", gb, first, outs[ip % 2].view(), wp)
        pending = (t, i, want)
    tp, ip, wp = pending
    gb.wait(tp)
    check_ticket(f"ticket {ip}", gb, first, outs[ip % 2].view(), wp)
    assert ga.counters() == gb.counters()
    for o in (wa, ga, wb, gb):
        o.close()


def test_interleaved_submit_and_process(gpu_ctx, tx):
    """submit, submit, process, submit, process (three times) gives what process alone gives; closing the front end with two
    tickets in flight leaves their host outputs complete"""
    import torch
    dab = gpu_ctx
    name = "k_wideband_s8"
    fs, _, _, offs, n_src, _ = CONFIGS[name]
    n_ch = n_src * len(offs)
    ga, wa, out_a = open_front_end(dab, tx, name)
    gb, wb, out_b = open_front_end(dab, tx, name)
    sizes = ticket_sizes(tx, fs, 17)
    max_n = max(sizes)
    wb.reserve(max_n)
    feed = Feed(tx, name, seed=6)
    itemsize = feed.raw.itemsize
    ins = [dab.HostBuffer(n_src * max_n * 2 * itemsize) for _ in range(2)]
    outs = [Outputs(dab, gb.P, n_ch) for _ in range(2)]
    pattern = "SSPSP" * 3 + "SS"
    in_flight = []
    for i, (m, kind) in enumerate(zip(sizes, pattern)):
        block = feed.next(m)
        wa.process(block, block_size=BLOCK)
        ga.chan_decode()
        want = serial_results(ga, 0, n_ch, 4)
        if kind == "P":
            wb.process(block, block_size=BLOCK)
            gb.chan_decode()
            got = serial_results(gb, 0, n_ch, 4, pop=False)
            for c, (w_c, g_c) in enumerate(zip(want, got)):
                assert w_c[0] == g_c[0] and np.array_equal(w_c[1], g_c[1]) and np.array_equal(w_c[2], g_c[2]), f"step {i} channel {c}"
                assert all(np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) for a, b in zip(w_c[3], g_c[3])), f"step {i} channel {c}"
            for t, j, wj in in_flight:
                gb.wait(t)
                check_ticket(f"ticket {j}", gb, 0, outs[j % 2].view(), wj, frames=False)
            in_flight = []
            continue
        if len(in_flight) == 2:   # both slots busy: retire the older ticket before its buffers are reused
            t, j, wj = in_flight.pop(0)
            gb.wait(t)
            check_ticket(f"ticket {j}", gb, 0, outs[j % 2].view(), wj, frames=False)
        ins[i % 2].array.view(block.dtype).reshape(n_src, max_n * 2)[:, :2 * m] = block
        outs[i % 2].poison()
        t = wb.submit(ins[i % 2].ptr.value, max_n * 2 * itemsize, m, block_size=BLOCK, run_chan_decode=True, **outs[i % 2].ptrs())
        in_flight.append((t, i, want))
    assert len(in_flight) == 2
    wb.close()   # returns once the copy-out of both tickets has finished
    for t, j, wj in in_flight:
        check_ticket(f"ticket {j} (closed in flight)", gb, 0, outs[j % 2].view(), wj, frames=False)
        gb.wait(t)
    torch.cuda.synchronize()
    assert torch.equal(out_a.view(torch.float32), out_b.view(torch.float32))
    assert ga.counters() == gb.counters()
    for o in (wa, ga, gb):
        o.close()


@pytest.mark.parametrize("name", list(CONFIGS))
def test_reserve_does_not_change_output(gpu_ctx, tx, name):
    import torch
    dab = gpu_ctx
    fs = CONFIGS[name][0]
    g1, w1, out1 = open_front_end(dab, tx, name)
    g2, w2, out2 = open_front_end(dab, tx, name)
    w2.reserve(3 * frame_input(tx, fs) + 12345)
    feed = Feed(tx, name, seed=7)
    for m in ticket_sizes(tx, fs, 9):
        block = feed.next(m)
        assert w1.process(block, block_size=BLOCK) == w2.process(block, block_size=BLOCK)
        torch.cuda.synchronize()
        assert torch.equal(out1.view(torch.float32), out2.view(torch.float32))
    assert g1.counters() == g2.counters()
    for o in (w1, g1, w2, g2):
        o.close()


def test_round_trip_32_sources_through_submit(gpu_ctx, tx):
    """32 sources x 4 ensembles at 8.192 MHz raw_s16l, one frame of input per ticket, two tickets in flight, nothing but submit:
    every channel gives back the transmitted logical frames in order (as test_wideband_gpu.round_trip requires), no RS,
    fire-code or AU-CRC failure, every FIB CRC good, no frame dropped"""
    dab = gpu_ctx
    D, fmt, rms = 4, "raw_s16l", 3000.0
    offs = [-2568000, -856000, 856000, 2568000]
    caps = [make_capture_pow2(tx, D, offs, [41 + 4 * u + k for k in range(4)], seed=4 + u) for u in range(2)]
    raws = [tx.quantize(cap, fmt, rms).reshape(-1, 2) for cap, _ in caps]
    FS = tx.MODES[1].nb_frame_samples
    source_map = [(s % 2, (s * 7919 * 37) % (PERIOD * FS * D)) for s in range(32)]
    channels = [(s, f, e) for s in range(32) for e, f in enumerate(offs)]
    subs = tx.default_ensemble()[:4]
    import torch
    n_ch = len(channels)
    g = dab.DabGpu(mode=1, max_streams=n_ch, iq_format=dab.IQ_C32)
    out = torch.zeros((n_ch, CAP), dtype=torch.complex64, device="cuda:0")
    w = g.wideband_open(D * 2048000, fmt, [c[0] for c in channels], [c[1] for c in channels], out.data_ptr(), CAP, n_sources=32)
    for c in range(n_ch):
        g.msc_configure(c, subs)
    layout = [g.msc_layout(0, k) for k in range(len(subs))]
    step = D * FS
    w.reserve(step)
    ins = [dab.HostBuffer(32 * step * 4, write_combined=True) for _ in range(2)]
    outs = [Outputs(dab, g.P, n_ch) for _ in range(2)]
    wts = np.random.default_rng(4).integers(1, 2 ** 63, size=256, dtype=np.uint64) | np.uint64(1)
    got = [[[] for _ in subs] for _ in range(n_ch)]
    c_start = None

    def collect(i):
        o = outs[i % 2].view()
        if i < WARM:
            return
        for c in np.nonzero(o["chan_status"][:, 0] == 1)[0]:
            assert o["fic_crc"][c, :, :3].all(), f"ticket {i}: channel {c}: a FIB failed its CRC"
            for k, (off, nb) in enumerate(layout):
                assert o["msc_valid"][c, :, k].all(), f"ticket {i}: channel {c} sub-channel {k}: a CIF is not valid"
                got[c][k].extend(_hash(o["msc"][c, :, off:off + nb], wts).tolist())

    pending = None
    n_tickets = WARM + 2 * PERIOD
    for i in range(n_tickets):
        if i == WARM:
            if pending is not None:
                g.wait(pending[0])
                collect(pending[1])
                pending = None
            c_start = g.counters()
        h = ins[i % 2].array.view(np.int16).reshape(32, 2 * step)
        for s, (ci, lead) in enumerate(source_map):
            h[s] = np.take(raws[ci], np.arange(lead + i * step, lead + (i + 1) * step), axis=0, mode="wrap").reshape(-1)
        t = w.submit(ins[i % 2].ptr.value, 2 * step * 2, step, block_size=BLOCK, run_chan_decode=True,
                     chan_status_host=outs[i % 2].bufs["chan_status"].ptr.value, msc_host=outs[i % 2].bufs["msc"].ptr.value,
                     msc_valid_host=outs[i % 2].bufs["msc_valid"].ptr.value, fic_crc_host=outs[i % 2].bufs["fic_crc"].ptr.value)
        if pending is not None:
            g.wait(pending[0])
            collect(pending[1])
        pending = (t, i)
    g.wait(pending[0])
    collect(pending[1])
    c_end = g.counters()
    d = {k: c_end[k] - c_start[k] for k in c_end}
    for c, (s, _, e) in enumerate(channels):
        logical = caps[source_map[s][0]][1][e]
        for k, sc in enumerate(subs):
            want = _hash(logical[sc.id], wts)
            seq = np.array(got[c][k], dtype=np.uint64)
            assert seq.size >= want.size, f"channel {c} sub-channel {k}: {seq.size} CIFs decoded in the window"
            j = np.nonzero(want == seq[0])[0]
            assert j.size == 1, f"channel {c} sub-channel {k}: decoded a logical frame that was not transmitted"
            assert np.array_equal(seq, want[(j[0] + np.arange(seq.size)) % want.size]), \
                f"channel {c} sub-channel {k}: decoded frames are not the transmitted ones in order, once per period"
    assert d["superframes_rs_fail"] == 0 and d["superframes_firecode_fail"] == 0 and d["au_crc_fail"] == 0
    assert d["fibs_crc_ok"] == d["fibs_total"] > 0 and d["frames_dropped"] == 0 and d["au_ok"] > 0
    w.close()
    g.close()


def test_errors(gpu_ctx):
    import torch
    dab = gpu_ctx
    out = torch.zeros((2, CAP), dtype=torch.complex64, device="cuda:0")
    g = dab.DabGpu(mode=1, max_streams=4, iq_format=dab.IQ_C32)
    w = g.wideband_open(8192000, "raw_s16l", [0, 1], [856000, -856000], out.data_ptr(), CAP)
    buf = dab.HostBuffer(2 * 4096 * 4)
    p = buf.ptr.value

    def rc(fn, *a, **k):
        try:
            fn(*a, **k)
        except dab.DabGpuError as e:
            return e.code, str(e)
        return dab.OK, ""

    code, msg = rc(w.submit, p, 4096 * 4, 1000)
    assert code == dab.ERR_INVALID and "reserve" in msg   # nothing reserved yet
    for bad in (0, 1 << 40):
        assert rc(w.reserve, bad)[0] == dab.ERR_INVALID
    w.reserve(2000)
    code, msg = rc(w.submit, p, 4096 * 4, 2001)
    assert code == dab.ERR_INVALID and "reserve" in msg
    for n in (0, -5):
        assert rc(w.submit, p, 4096 * 4, n)[0] == dab.ERR_INVALID
    assert rc(w.submit, p, 2000 * 4 - 1, 2000)[0] == dab.ERR_INVALID   # stride shorter than a source
    assert rc(w.submit, 0, 4096 * 4, 1000)[0] == dab.ERR_INVALID
    for first, n in ((-1, 1), (0, 3), (2, 1), (1, 2), (0, 0)):
        assert rc(w.submit, p, 4096 * 4, 1000, first_stream=first, n_streams=n)[0] == dab.ERR_INVALID, (first, n)
    g.wait(w.submit(p, 4096 * 4, 2000, first_stream=1, n_streams=1, run_chan_decode=True))
    assert rc(w.reserve, 4000)[0] == dab.ERR_STATE   # input was fed
    assert rc(g.submit, p, 4096 * 2, 1000)[0] == dab.ERR_STATE   # dabgpu_submit while the front end is attached
    assert w.process(np.zeros((2, 2 * 1000), dtype=np.int16)) >= 0   # process may follow submit
    g.L.dabgpu_ctx_destroy(g.h)
    g.h, g._wideband = None, None
    assert rc(w.submit, p, 4096 * 4, 1000)[0] == dab.ERR_STATE
    assert rc(w.reserve, 1000)[0] == dab.ERR_STATE
    w.close()
