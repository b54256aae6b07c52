"""Oracle of the packet-mode sub-channel stage (DABGPU_PAYLOAD_PACKET / _PACKET_FEC) and the stream scenarios shared by its tests.

PacketOracle is oracle/pyref.py:PortPacketFec (pinned to the reference's callback log by test_packet_fec_cpu.py) with the
records the channel decode reports: every callback becomes a PACKET record (is_corrected, crc_ok, address), every end of a
set a PACKET_FEC record (decoded, rows decoded, rows uncorrectable, sum of the decoded rows' error counts) just before the
packets it releases.  A logical frame is walked the way basic_data_packet_channel.cpp:49-88 walks it."""
import struct

import numpy as np

EV_PACKET, EV_PACKET_FEC = 6, 7
FEC_ADDRESS = 1022


def crc_ok(tx, p: bytes) -> int:
    a = np.frombuffer(p, dtype=np.uint8)
    return int(tx.crc16_ccitt(a[:-2]) == (int(a[-2]) << 8 | int(a[-1])))


def address(p: bytes) -> int:
    return ((p[0] & 3) << 8) | p[1]


def record(kind, a, b, c, d, payload=b"") -> bytes:
    return struct.pack("<6i", kind, a, b, c, d, len(payload)) + payload


def parse(log: bytes):
    """sub-channel event log -> [(type, a, b, c, d, payload)]"""
    out, off = [], 0
    while off < len(log):
        t, a, b, c, d, n = struct.unpack_from("<6i", log, off)
        off += 24
        out.append((t, a, b, c, d, bytes(log[off:off + n])))
        off += (n + 3) & ~3
    return out


def make_oracle(pyref, tx, fec: bool):
    class PacketOracle(pyref.PortPacketFec):
        def __init__(self):
            super().__init__()
            self.fec_mode = fec
            self.events = []       # PACKET_FEC fields of the sets ended by the last read_packet, in order
            self._pending = []

        def _clear(self, out):
            self._pending.append((len(out), (0, 0, 0, 0)))
            super()._clear(out)

        def _correct(self, out):
            # PortPacketFec._correct with the row counts kept
            at = lambda off: (self.rd + off) % self.RING
            table = np.zeros(192, dtype=np.uint8)
            for i in range(9):
                n = 22 if i < 8 else 16
                table[22 * i:22 * i + n] = self.ring[[at(2256 + 24 * i + 2 + j) for j in range(n)]]
            ok = bad = total = 0
            for y in range(12):
                cw = np.concatenate([self.ring[[at(12 * x + y) for x in range(188)]], table[[12 * i + y for i in range(16)]]])
                cnt, fixed, pos = self.rs.decode(cw)
                if cnt < 0:
                    bad += 1
                    continue
                ok += 1
                total += cnt
                for p in pos[:cnt]:
                    x = int(p) - 51
                    if 0 <= x < 188:
                        self.ring[at(12 * x + y)] = fixed[x]
            self._pending.append((len(out), (1, ok, bad, total)))
            n0 = len(out)
            total_bytes = 0
            while total_bytes < 2256:
                p = self._pop()
                if p is None:
                    break
                out.append((p, True))
                total_bytes += len(p)
            assert n0 == self._pending[-1][0]

        def read_records(self, buf) -> tuple:
            """-> (bytes consumed, records) of one ReadPacket call"""
            self._pending = []
            buf = np.asarray(buf, dtype=np.uint8)
            if self.fec_mode:
                used, out = self.read_packet(buf)
            else:
                used, out = self._plain(buf)
            recs, k = [], 0
            for i, (p, corrected) in enumerate(out):
                while k < len(self._pending) and self._pending[k][0] == i:
                    recs.append(record(EV_PACKET_FEC, *self._pending[k][1]))
                    k += 1
                recs.append(record(EV_PACKET, int(corrected), crc_ok(tx, p), address(p), 0, p))
            for _, f in self._pending[k:]:
                recs.append(record(EV_PACKET_FEC, *f))
            return used, recs

        @staticmethod
        def _plain(buf):
            if buf.size < 2:
                return int(buf.size), []
            n = 24 * ((int(buf[0]) >> 6) + 1)
            if buf.size < n:
                return int(buf.size), []
            return n, [(bytes(buf[:n]), False)]

        def frame(self, frame) -> bytes:
            """one logical frame walked as the channel does -> the records (log bytes)"""
            frame = np.asarray(frame, dtype=np.uint8)
            pos, log = 0, b""
            while pos < frame.size:
                used, recs = self.read_records(frame[pos:])
                log += b"".join(recs)
                pos += used
            return log

    return PacketOracle()


# ---- transmitter hooks realising the scenarios of tests/golden/make_packet_fec_golden.py on a packet stream ----------------
def _flip(rng, p, lo=2):
    p[int(rng.integers(lo, p.size))] ^= int(rng.integers(1, 256))


def scenario_hook(tx, seed: int):
    """packet_hook cycling through: clean; byte errors every row can correct; errors beyond the code; a lost packet; a broken
    FEC counter; an extra packet (eviction); header errors; FEC packets whose length field claims 96 bytes.  Only FEC sets
    (batches ending in the nine FEC packets) are touched."""
    rng = np.random.default_rng(seed)
    count = [0]

    def hook(sc, pkts):
        if not sc.packet_fec:
            if rng.random() < 0.2 and pkts:
                _flip(rng, pkts[int(rng.integers(0, len(pkts)))], 0)
            return pkts
        k = count[0] % 8
        count[0] += 1
        pkts = [p.copy() for p in pkts]
        data = pkts[:-9]
        if k == 1:
            flat = np.concatenate(data)
            for y in range(12):
                x = rng.choice(188, size=3, replace=False)
                flat[12 * x + y] ^= rng.integers(1, 256, 3, dtype=np.uint8)
            off = 0
            for p in data:
                keep = p[0] & 0xC0
                p[:] = flat[off:off + p.size]
                p[0] = (p[0] & 0x3F) | keep
                off += p.size
        elif k == 2:
            for _ in range(60):
                _flip(rng, data[int(rng.integers(0, len(data)))])
            data[0][2:] ^= 0x5A
        elif k == 3:
            del pkts[int(rng.integers(0, len(data)))]
        elif k == 4:
            pkts[-4][0] ^= 0x04
        elif k == 5:
            pkts = [rng.integers(0, 256, 24, dtype=np.uint8) & np.uint8(0x3F)] + pkts
        elif k == 6:
            for _ in range(8):
                p = data[int(rng.integers(0, len(data)))]
                p[int(rng.integers(1, p.size))] ^= int(rng.integers(1, 256))
        elif k == 7:
            for p in pkts[-9:]:
                p[0] |= 0xC0
        return pkts

    return hook
