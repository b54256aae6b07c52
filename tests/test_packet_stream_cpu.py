"""Packet-mode sub-channels, CPU side: the transmitter's packet streams (synth/dabtx.py) and the oracle of the channel decode's
packet records (tests/packet_cases.py), which is PortPacketFec plus the CRC flag and the PACKET_FEC fields."""
import os

import numpy as np

import packet_cases as pc
from conftest import GOLDEN


def _ensemble(tx, hook=None, seed=11):
    subs = [tx.Subchannel(0, 0, 48),
            tx.Subchannel(1, 48, 12, eep_level=0, packet_fec=True),            # 8 kbit/s: a set spans many frames
            tx.Subchannel(2, 60, 72, eep_level=1, packet_fec=True),            # 96 kbit/s
            tx.Subchannel(3, 132, 18, eep_level=1, packet_fec=False)]
    return subs, tx.EnsembleTx(1, subs, seed=seed, packet_hook=hook)


def _frames(tx, n_frames, hook=None):
    subs, ens = _ensemble(tx, hook)
    for _ in range(n_frames):
        ens.next_frame_bits()
    return subs, ens


def test_transmitted_packets_are_valid(tx):
    subs, ens = _frames(tx, 40)
    for sc in subs[1:]:
        pk = ens.packets[sc.id]
        assert len(pk) > 20
        for p in pk:
            assert p.size in (24, 48, 72, 96)
            if pc.address(p.tobytes()) != pc.FEC_ADDRESS:
                assert pc.crc_ok(tx, p.tobytes()), sc.id
                assert (p[2] & 0x7F) <= p.size - 5
        frames = np.concatenate(ens.logical_frames[sc.id])
        assert all(f.size % 24 == 0 for f in ens.logical_frames[sc.id])
        # the stream is the packets back to back, whole packets in every logical frame
        sent = np.concatenate(pk)
        n = min(sent.size, frames.size)
        assert np.array_equal(sent[:n], frames[:n])
        addrs = {pc.address(p.tobytes()) for p in pk} - {0, pc.FEC_ADDRESS}
        assert addrs and all(1 + 3 * sc.id <= a < 4 + 3 * sc.id for a in addrs)
    fec = [p for p in ens.packets[2] if pc.address(p.tobytes()) == pc.FEC_ADDRESS]
    assert len(fec) % 9 == 0 and len(fec) >= 18


def test_port_processor_returns_every_transmitted_packet(pyref, tx):
    subs, ens = _frames(tx, 40)
    for sc in subs[1:]:
        port = pyref.PortPacketFec()
        got = []
        for f in ens.logical_frames[sc.id]:
            pos = 0
            while pos < f.size:
                used, out = port.read_packet(f[pos:]) if sc.packet_fec else (24 * ((int(f[pos]) >> 6) + 1), [(f[pos:pos + 24 * ((int(f[pos]) >> 6) + 1)].tobytes(), False)])
                got += out
                pos += used
        data = [p.tobytes() for p in ens.packets[sc.id] if pc.address(p.tobytes()) != pc.FEC_ADDRESS]
        assert [p for p, _ in got] == data[:len(got)]
        if sc.packet_fec:
            assert all(ok for _, ok in got) and len(got) >= len(data) - 2256 // 24
        else:
            assert len(got) == len(data)


def test_oracle_records_match_golden_callbacks(pyref, tx):
    """the oracle's PACKET records, stripped to (packet, is_corrected), are the reference's callbacks call by call; crc_ok and
    the address are those of the packet; every set end gives one PACKET_FEC record"""
    kat = np.load(os.path.join(GOLDEN, "packet_fec_kat.npz"))
    off = np.concatenate([[0], np.cumsum(kat["call_len"])])
    loff = np.concatenate([[0], np.cumsum(kat["log_len"])])
    o = pc.make_oracle(pyref, tx, fec=True)
    n_fec = {0: 0, 1: 0}
    for i in range(kat["call_len"].size):
        used, recs = o.read_records(kat["calls"][off[i]:off[i + 1]])
        assert used == int(kat["used"][i])
        ev = pc.parse(b"".join(recs))
        exp = pyref.parse_packet_log(kat["logs"][loff[i]:loff[i + 1]].tobytes())
        assert [(p, bool(a)) for t, a, b, c, d, p in ev if t == pc.EV_PACKET] == exp, f"call {i}"
        for t, a, b, c, d, p in ev:
            if t == pc.EV_PACKET:
                assert b == pc.crc_ok(tx, p) and c == pc.address(p) and d == 0
            else:
                assert t == pc.EV_PACKET_FEC and p == b""
                n_fec[a] += 1
                assert (b + c == 12 and d >= 0) if a else (b, c, d) == (0, 0, 0)
        # a set that ends releases its packets right behind its PACKET_FEC record
        if any(t == pc.EV_PACKET_FEC for t, *_ in ev):
            assert ev[0][0] == pc.EV_PACKET_FEC
    assert n_fec[1] >= 5 and n_fec[0] >= 3


def test_hook_scenarios_reach_every_exit(pyref, tx):
    """the scenario hook used on the GPU drives the processor through corrected sets, failed rows, abandoned sets and evictions"""
    subs, ens = _frames(tx, 130, pc.scenario_hook(tx, 5))
    o = pc.make_oracle(pyref, tx, fec=True)
    ev = []
    for f in ens.logical_frames[2]:
        ev += pc.parse(o.frame(f))
    fec = [e for e in ev if e[0] == pc.EV_PACKET_FEC]
    assert any(e[1] == 1 and e[3] == 0 and e[4] > 0 for e in fec)      # corrected errors
    assert any(e[1] == 1 and e[3] > 0 for e in fec)                     # rows beyond the code
    assert any(e[1] == 0 for e in fec)                                  # abandoned sets
    pk = [e for e in ev if e[0] == pc.EV_PACKET]
    assert any(e[1] == 0 for e in pk) and any(e[1] == 1 for e in pk) and any(e[2] == 0 for e in pk)


def test_new_symbols_exported(dab):
    L = dab.load_library()
    for name in ("dabgpu_msc_configure_ex", "dabgpu_msc_add_subchannel_ex"):
        assert hasattr(L, name) and name in dab.EXPORTS
    assert (dab.EV_PACKET, dab.EV_PACKET_FEC) == (pc.EV_PACKET, pc.EV_PACKET_FEC)
    assert (dab.PAYLOAD_STREAM, dab.PAYLOAD_DABPLUS, dab.PAYLOAD_PACKET, dab.PAYLOAD_PACKET_FEC) == (0, 1, 2, 3)
