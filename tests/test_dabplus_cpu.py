"""The DAB+ superframe cases of tests/dabplus_cases.py checked against the C restatement of AAC_Frame_Processor: each case makes
the oracle emit exactly the events it is meant to, so a GPU mismatch on these cases is the kernel's fault.  No GPU needed."""
import numpy as np
import pytest

import dabplus_cases as dc


def expected(pyref, s: dc.Superframe) -> list:
    """events of a superframe decoded while synced, as (type, a, b, payload) -- c/d (received / computed CRC) left out"""
    if s.rs_fail is not None:
        return [(pyref.EV_RS_ERROR, s.rs_fail, s.N, b"")]
    if s.bad_fire:
        return [(pyref.EV_FIRECODE_ERROR, 5, int(s.sf[0]) << 8 | int(s.sf[1]), b"")]
    d = s.dsc
    n_aus = dc.N_AUS[((d >> 6) & 1, (d >> 5) & 1)]
    out = [(pyref.EV_HEADER, 48000 if d & 0x40 else 32000, ((d >> 3) & 1) | ((d >> 4) & 2) | ((d >> 2) & 4), b"")]
    for i, p in enumerate(s.payloads):
        out.append((pyref.EV_AU_CRC_ERROR, i, n_aus, b"") if i in s.bad_crc else (pyref.EV_AU, i, n_aus, p))
    return out


def feed(aac, s: dc.Superframe) -> list:
    evs = []
    for k, fr in enumerate(s.frames()):
        got = aac.process(fr)
        assert k == 4 or not got, (k, got)
        evs += got
    return evs


@pytest.mark.parametrize("layout", dc.LAYOUTS, ids=lambda l: f"dac{l[0]}-sbr{l[1]}")
@pytest.mark.parametrize("N", list(range(1, 25)) + [32, 48, 96, 288])
def test_cases_make_the_oracle_emit_what_they_intend(tx, pyref, N, layout):
    rng = np.random.default_rng(1000 * N + 10 * layout[0] + layout[1])
    aac, rs = pyref.PortAac(), pyref.PortRS()
    prog = dc.program(tx, rng, N, *layout, mpeg=(0, 1, 2, 7, 5)[N % 5], rs_fails=lambda cw: rs.decode(cw)[0] < 0)
    labels = set()
    for s in prog:
        evs = feed(aac, s)
        got = [(t, a, b, p) for t, a, b, c, d, p in evs]
        exp = expected(pyref, s)
        assert got == exp, f"N={N} dac_rate/sbr={layout} case '{s.label}': {[e[:3] for e in got]} != {[e[:3] for e in exp]}"
        labels.add(s.label)
    kinds = {s.label.split(" ")[0] for s in prog}
    assert len(prog) >= 14 and {"even", "longest", "fire", "6", "12"} <= kinds, (N, layout, sorted(labels))
    if N >= 20 and layout == (0, 1):
        assert {"2114-byte AU 0", "2115-byte AU 0", "2153-byte AU 0"} <= labels


def test_au_lengths_and_starts(tx, pyref):
    """the builder lays out what it is asked for: AU lengths, empty AUs, the longest AU, starts beyond the end"""
    rng = np.random.default_rng(7)
    s = dc.build(tx, rng, 20, dac_rate=0, sbr=1, starts=dc.split_starts(20, 2, [2153]))
    assert [n for _, n in s.aus] == [2153, 2200 - 5 - 2153 - 4]
    s = dc.build(tx, rng, 288, dac_rate=1, sbr=0, starts=[3992] * 4 + [4000])
    assert [n for _, n in s.aus] == [3992 - 11 - 2]     # AU 1 = [3992, 3992) is out of bounds: the walk stops
    s = dc.build(tx, rng, 288, dac_rate=0, sbr=1, starts=[4000])
    assert [n for _, n in s.aus] == [4000 - 5 - 2, 110 * 288 - 4000 - 2]
    s = dc.build(tx, rng, 8, dac_rate=1, sbr=1, starts=[100, 4095])
    assert [n for _, n in s.aus] == [100 - 6 - 2]
    evs = feed(pyref.PortAac(), s)
    assert [e[0] for e in evs] == [pyref.EV_HEADER, pyref.EV_AU]


@pytest.mark.parametrize("n", [0, 1, 5, 10, 11, 23, 25, 121, 1001, 4801])
def test_frame_lengths_not_multiple_of_24(tx, pyref, n):
    """odd frame lengths: N = 5 n // 120 codewords, the rest unprotected; below 11 bytes the processor ignores the frame"""
    rng = np.random.default_rng(n)
    aac = pyref.PortAac()
    if n < 11:
        for _ in range(6):
            assert aac.process(rng.integers(0, 256, size=n, dtype=np.uint8)) == []
        return
    N = 5 * n // 120
    starts = [min(dc.header_len(2) + 2 + max(110 * N - 7, 0) // 3, dc.AU_START_MAX)] if N else [5 * n - 1]
    s = dc.build(tx, rng, frame_bytes=n, dac_rate=0, sbr=1, starts=starts)
    evs = feed(aac, s)
    assert [e[0] for e in evs] == [pyref.EV_HEADER] + [pyref.EV_AU] * len(s.aus), (n, [e[:3] for e in evs])
    assert [e[5] for e in evs[1:]] == s.payloads
