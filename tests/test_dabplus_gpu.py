"""DAB+ superframe stage on the GPU against the oracle: the stand-alone processor (dabgpu_dabplus_process, k_dabplus_direct) and
the batched stage after the MSC decoder (k_dabplus), at every superframe size, AU layout and error pattern of
tests/dabplus_cases.py.

Bar: the event log of every frame (direct) or of every (stream, sub-channel) per decode call (batched) is byte-identical to
the oracle's, and the context counters move by the oracle's event counts."""
import numpy as np
import pytest

import dabplus_cases as dc

pytestmark = pytest.mark.gpu

SIZES = list(range(1, 25)) + [32, 48, 96, 288]     # 6912-byte frames (N = 288) are the largest a sub-channel can have


def _aac(pyref):
    return pyref.RefAac() if pyref.ref_available() else pyref.PortAac()


def _counts(pyref, events) -> dict:
    """what each context counter must have advanced by for these oracle events"""
    t = [e[0] for e in events]
    return {"superframes_ok": t.count(pyref.EV_HEADER), "superframes_rs_fail": t.count(pyref.EV_RS_ERROR),
            "superframes_firecode_fail": sum(1 for e in events if e[0] == pyref.EV_FIRECODE_ERROR and e[1] == 5),
            "au_crc_fail": t.count(pyref.EV_AU_CRC_ERROR), "au_ok": t.count(pyref.EV_AU)}


def _delta(g, c0) -> dict:
    c1 = g.counters()
    return {k: c1[k] - c0[k] for k in ("superframes_ok", "superframes_rs_fail", "superframes_firecode_fail", "au_crc_fail", "au_ok")}


def _run_direct(g, pyref, frames, what: str) -> list:
    """frames: [(label, bytes)] fed to one new processor and one new oracle; returns the oracle's events"""
    proc, aac, c0, events = g.dabplus_open(), _aac(pyref), g.counters(), []
    try:
        for k, (label, fr) in enumerate(frames):
            exp = aac.process(fr)
            got = g.dabplus_process(proc, fr)
            assert got == dc.event_log(exp), \
                f"{what}, frame {k} ({fr.size} bytes, {label}): {[e[:5] for e in pyref.parse_event_log(got)]} != {[e[:5] for e in exp]}"
            events += exp
    finally:
        g.dabplus_close(proc)
    assert _delta(g, c0) == _counts(pyref, events), what
    return events


def _frames(superframes) -> list:
    return [(f"{s.label}, logical frame {k}", fr) for s in superframes for k, fr in enumerate(s.frames())]


@pytest.mark.parametrize("N", SIZES)
def test_direct_every_layout_and_error_pattern(gpu_ctx, tx, pyref, N):
    """The programs test_dabplus_cpu.py checks against the oracle (same seeds): every AU layout, AU lengths 0 .. 110 N - 9
    incl. both sides of 2115 bytes, AU CRC / fire-code failures, RS errors in every position and pass, AU-start tables the
    header walk stops at.  mpeg cycles through 0, 1, 2, 7, 5 with N."""
    g = gpu_ctx.DabGpu(mode=1, max_streams=1)
    rs = pyref.PortRS()
    kinds = set()
    for layout in dc.LAYOUTS:
        rng = np.random.default_rng(1000 * N + 10 * layout[0] + layout[1])
        prog = dc.program(tx, rng, N, *layout, mpeg=(0, 1, 2, 7, 5)[N % 5], rs_fails=lambda cw: rs.decode(cw)[0] < 0)
        events = _run_direct(g, pyref, _frames(prog), f"N={N} dac_rate/sbr={layout}")
        kinds |= {e[0] for e in events}
    assert kinds == {pyref.EV_HEADER, pyref.EV_AU, pyref.EV_AU_CRC_ERROR, pyref.EV_RS_ERROR, pyref.EV_FIRECODE_ERROR}, (N, kinds)
    g.close()


@pytest.mark.parametrize("N", [8, 20])
def test_direct_sync_state_machine(gpu_ctx, tx, pyref, N):
    """Garbage before sync, fire-code errors while searching, ten failing superframes in a row (the processor drops sync and
    searches again) and resync, a change of frame length in the middle of a superframe."""
    rng = np.random.default_rng(50 + N)
    rs = pyref.PortRS()
    g = gpu_ctx.DabGpu(mode=1, max_streams=1)
    good = lambda n=N, **kw: dc.build(tx, rng, n, **kw)
    base = good()
    rs_fail = base.with_errors(dc.cw_errors(rng, N - 1, 30), "30 errors in codeword N-1")
    assert rs.decode(rs_fail.sf[N - 1::N][:120])[0] < 0
    frames = [("garbage", rng.integers(0, 256, size=24 * N, dtype=np.uint8)) for _ in range(3)]
    frames += _frames([good(bad_fire=True, label="fire code while searching"), good(label="sync"), good(label="synced")])
    frames += _frames([rs_fail if i % 2 else good(bad_fire=True, label=f"failing superframe {i}") for i in range(10)])
    frames += [("garbage after 10 failures", rng.integers(0, 256, size=24 * N, dtype=np.uint8))]
    frames += _frames([good(label="resync"), good(label="synced")])
    frames += _frames([rs_fail] * 10 + [good(label="resync after 10 RS failures")])
    frames += _frames([good()])[:2]
    frames += _frames([good(N + 2, label="frame length change"), good(N + 2, dac_rate=0, sbr=0)])
    frames += _frames([good(N + 2)])[:3] + _frames([good(label="back to the first length"), good(dac_rate=1, sbr=0)])
    events = _run_direct(g, pyref, frames, f"N={N} sync sequence")
    fire = [e for e in events if e[0] == pyref.EV_FIRECODE_ERROR]
    assert {e[1] for e in fire} == {0, 5} and sum(e[0] == pyref.EV_HEADER for e in events) >= 8
    g.close()


@pytest.mark.parametrize("n", [11, 23, 25, 121, 1001, 4801])
def test_direct_frame_lengths_not_multiple_of_24(gpu_ctx, tx, pyref, n):
    """Odd logical frame lengths (the unaligned copy and global-memory superframe paths; N = 5 n // 120 codewords, the rest of
    the 5 n bytes unprotected).  Frames shorter than 11 bytes, interleaved, must produce nothing and leave the state alone."""
    rng = np.random.default_rng(n)
    g = gpu_ctx.DabGpu(mode=1, max_streams=1)
    N = 5 * n // 120
    sfs = []
    for dac_rate, sbr in dc.LAYOUTS:
        n_aus = dc.N_AUS[(dac_rate, sbr)]
        hdr = dc.header_len(n_aus)
        if N:
            starts = [min(hdr + (i + 1) * max(110 * N - hdr, 0) // n_aus, dc.AU_START_MAX) for i in range(n_aus - 1)]
        else:   # no codeword: AUs may sit anywhere before the end, the last one (ending at 110 N = 0) is out of bounds
            starts = [hdr + (i + 1) * (5 * n - hdr) // n_aus for i in range(n_aus - 1)]
        kw = dict(frame_bytes=n, dac_rate=dac_rate, sbr=sbr, starts=starts)
        sfs += [dc.build(tx, rng, label=f"dac_rate/sbr={dac_rate, sbr}", **kw), dc.build(tx, rng, bad_crc=(0,), label="AU 0 CRC", **kw)]
        if N:
            base = sfs[-2]
            sfs.append(base.with_errors(dc.cw_errors(rng, N - 1, 5), "5 errors in codeword N-1"))
            sfs.append(base.with_errors(dc.cw_errors(rng, 0, 9), "9 errors in codeword 0"))
    frames = []
    for k, item in enumerate(_frames(sfs)):
        frames.append(item)
        if k % 3 == 1:
            m = (0, 1, 5, 10)[k % 4]
            frames.append((f"{m}-byte frame", rng.integers(0, 256, size=m, dtype=np.uint8)))
    events = _run_direct(g, pyref, frames, f"{n}-byte frames")
    assert sum(e[0] == pyref.EV_AU for e in events) >= 4
    g.close()


def _batched_subs(tx):
    """EEP 4-A (4 CU per 8 kbit/s) at N = 1 .. 24, 3-A for N = 2 (type-A sub-channels of 8 CU decode only 24 bytes), and 4-B
    at N = 8: 542 of the 864 CU."""
    subs, start = [], 0
    for i, N in enumerate((1, 2, 3, 5, 7, 8, 9, 15, 16, 17, 20, 24)):
        subs.append(tx.Subchannel(i, start, 12, eep_level=2) if N == 2 else tx.Subchannel(i, start, 4 * N, eep_level=3))
        start += subs[-1].length
    subs.append(tx.Subchannel(12, start, 30, eep_level=3, eep_type_b=True))
    return subs


def test_batched_every_size_with_errors(gpu_ctx, tx, pyref, monkeypatch):
    """k_dabplus through msc_configure -> softbits_push -> chan_decode: three streams (the last with 7 of the 13
    sub-channels, so the persistent CTAs meet empty items), one call covering streams 1-2 and one covering stream 0 only.
    The transmitter's superframes are replaced by cases picked by bitrate and count: every AU layout, AUs of 2115 bytes and
    more, AU CRC failures, uncorrectable codewords in a later pass, fire-code failures."""
    subs = _batched_subs(tx)
    for sc in subs:
        assert sc.frame_bytes % 24 == 0 and sc.frame_bytes // 24 in (1, 2, 3, 5, 7, 8, 9, 15, 16, 17, 20, 24), sc
    assert sum(sc.length for sc in subs) == 542
    rs = pyref.PortRS()
    count, labels = {}, {}

    def fake_superframe(bitrate_kbps, rng, **_):
        N = bitrate_kbps // 8
        k = count[N] = count.get(N, -1) + 1
        dac_rate, sbr = dc.LAYOUTS[(k // 6) % 4]
        n_aus = dc.N_AUS[(dac_rate, sbr)]
        kw = dict(dac_rate=dac_rate, sbr=sbr, mpeg=(0, 1, 2, 7, 3)[k % 5], label=f"N={N} dac_rate/sbr={dac_rate, sbr}")
        case = k % 6
        if case == 1:
            s = dc.build(tx, rng, N, starts=dc.split_starts(N, n_aus, [0] * (n_aus - 1)), **kw)
            s.label += f", longest last AU ({s.aus[-1][1]} bytes)"
        elif case == 2:
            s = dc.build(tx, rng, N, bad_crc=(k % n_aus,), **kw)
            s.label += f", AU {k % n_aus} CRC"
        elif case == 3:
            s = dc.build(tx, rng, N, **kw)
            while True:
                errs = dc.cw_errors(rng, N - 1, 7)
                t = s.with_errors(errs, s.label + f", 7 errors in codeword {N - 1}")
                if rs.decode(t.sf[N - 1:120 * N:N])[0] < 0:
                    break
            s = t.with_errors(dc.cw_errors(rng, 0, 5), t.label + ", 5 in codeword 0")
        elif case == 4:
            s = dc.build(tx, rng, N, bad_fire=True, **kw)
            s.label += ", fire code"
        elif case == 5 and dc.header_len(n_aus) + 2117 + k % 3 + 2 * (n_aus - 1) <= 110 * N:
            s = dc.build(tx, rng, N, starts=dc.split_starts(N, n_aus, [2115 + k % 3] + [0] * (n_aus - 2)), **kw)
            s.label += f", {2115 + k % 3}-byte AU 0"
        else:
            s = dc.build(tx, rng, N, **kw)
            s = s.with_errors(sum((dc.cw_errors(rng, cw, 5) for cw in range(0, N, 3)), []), s.label + ", 5 errors in every third codeword")
        labels[id(s.sf)] = s.label
        return s.sf

    monkeypatch.setattr(tx, "build_superframe", fake_superframe)
    n_streams = 3
    stream_subs = [subs, subs, subs[:7]]
    enss = [tx.EnsembleTx(1, stream_subs[s], seed=300 + 7 * s) for s in range(n_streams)]
    g = gpu_ctx.DabGpu(mode=1, max_streams=n_streams)
    for s in range(n_streams):
        g.msc_configure(s, stream_subs[s])
    aacs = [[_aac(pyref) for _ in stream_subs[s]] for s in range(n_streams)]
    seen = [[0] * len(stream_subs[s]) for s in range(n_streams)]
    c0, events = g.counters(), []
    for f in range(30):
        first, n = {12: (1, 2), 21: (0, 1)}.get(f, (0, n_streams))
        frames = np.stack([tx.hard_to_soft(enss[s].next_frame_bits()) for s in range(first, first + n)])
        g.softbits_push(frames, first_stream=first)
        g.chan_decode(first, n)
        for s in range(first, first + n):
            assert g.chan_status(s)[0] == 1, (f, s)
            for k, sc in enumerate(stream_subs[s]):
                out, valid = g.get_msc(s, k)
                log, j0 = b"", seen[s][k]
                for c in range(4):
                    if not valid[c]:
                        continue
                    sent = enss[s].logical_frames[sc.id][seen[s][k]]
                    assert np.array_equal(out[c], sent), f"frame {f} stream {s} sub-channel {k} CIF {c}: MSC bytes differ from those sent"
                    seen[s][k] += 1
                    exp = aacs[s][k].process(out[c])
                    events += exp
                    log += dc.event_log(exp)
                got = g.get_dabplus_events(s, k)
                cases = [labels[id(sf)] for sf in enss[s].superframes[sc.id][j0 // 5:(seen[s][k] + 4) // 5]]
                assert got == log, (f"frame {f} stream {s} sub-channel {k} ({cases}): "
                                    f"{[e[:5] for e in pyref.parse_event_log(got)]} != {[e[:5] for e in pyref.parse_event_log(log)]}")
    assert _delta(g, c0) == _counts(pyref, events)
    kinds = {e[0] for e in events}
    assert kinds == {pyref.EV_HEADER, pyref.EV_AU, pyref.EV_AU_CRC_ERROR, pyref.EV_RS_ERROR, pyref.EV_FIRECODE_ERROR}, kinds
    assert any(e[0] == pyref.EV_RS_ERROR and e[1] >= 8 for e in events), "no uncorrectable codeword in a later pass"
    assert any(e[0] == pyref.EV_AU and len(e[5]) >= 2115 for e in events), "no AU of 2115 bytes or more"
    g.close()
