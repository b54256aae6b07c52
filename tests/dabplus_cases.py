"""Shared by the DAB+ superframe tests: superframes of any size with an explicit access-unit (AU) layout, built with the
transmitter's CRC, fire code and RS(120,110) encoder, and the corruptions the superframe stage must tell apart.

N is the number of RS codewords of a superframe (bitrate / 8 kbit/s); a superframe is 120 N bytes sent as 5 logical frames of
24 N bytes, codeword i = bytes {i + j N}.  Frames of other lengths n give N = 5 n // 120 and 5 n - 120 N unprotected bytes."""
import numpy as np

N_AUS = {(0, 1): 2, (1, 1): 3, (0, 0): 4, (1, 0): 6}    # (dac_rate, sbr) -> access units per superframe
LAYOUTS = tuple(N_AUS)
AU_START_MAX = 4095                                       # the AU-start table holds 12-bit values


def header_len(n_aus: int) -> int:
    """fire code (2) + header byte + the 12-bit starts of AUs 1 .. n_aus-1: where AU 0 begins"""
    return 3 + (12 * (n_aus - 1) + 7) // 8


def even_starts(N: int, n_aus: int) -> list:
    """build_superframe's even split, squeezed under the 12-bit limit for N > 37 (the last AU then takes the rest)"""
    hdr = header_len(n_aus)
    base = (110 * N - hdr) // n_aus
    if n_aus > 1:
        base = min(base, (AU_START_MAX - hdr) // (n_aus - 1))
    return [hdr + i * base for i in range(1, n_aus)]


def split_starts(N: int, n_aus: int, lengths) -> list:
    """AU-start table for AUs 0 .. n_aus-2 of the given payload lengths (CRC not counted); the last AU ends at 110 N"""
    starts, pos = [], header_len(n_aus)
    for n in lengths[:n_aus - 1]:
        pos += n + 2
        starts.append(pos)
    assert pos + 2 <= 110 * N and pos <= AU_START_MAX, (N, n_aus, lengths)
    return starts


class Superframe:
    """sf: the 5 * frame_bytes bytes as sent; aus: [(start, payload length)] of the AUs the decoder should accept, in order,
    ending where its header walk stops ("access unit out of bounds").  label says what the case is; rs_fail is the first
    codeword the case makes uncorrectable (None: RS repairs every codeword)."""

    def __init__(self, sf: np.ndarray, frame_bytes: int, aus: list, label: str = "", bad_crc=(), bad_fire: bool = False):
        self.sf, self.frame_bytes, self.aus = sf, frame_bytes, aus
        self.label, self.bad_crc, self.bad_fire, self.rs_fail = label, tuple(bad_crc), bad_fire, None
        # header byte and AU payloads as built, before any byte error
        self.dsc, self.payloads = int(sf[2]), [bytes(sf[a:a + n]) for a, n in aus]

    @property
    def N(self) -> int:
        return 5 * self.frame_bytes // 120

    def with_errors(self, errors, label: str, rs_fail=None) -> "Superframe":
        """a copy with (codeword, position, xor value) byte errors made after the parity, position 0 .. 119"""
        out = Superframe(self.sf.copy(), self.frame_bytes, self.aus, label, self.bad_crc, self.bad_fire)
        out.dsc, out.payloads = self.dsc, self.payloads
        for cw, pos, v in errors:
            assert 0 <= cw < self.N and 0 <= pos < 120 and v
            out.sf[cw + pos * self.N] ^= v
        out.rs_fail = rs_fail
        return out

    def frames(self) -> list:
        return [self.sf[k * self.frame_bytes:(k + 1) * self.frame_bytes].copy() for k in range(5)]


def build(tx, rng, N: int = 0, frame_bytes: int = 0, dac_rate: int = 1, sbr: int = 1, stereo: int = 1, ps: int = 0, mpeg: int = 0,
          starts=None, bad_crc=(), bad_fire: bool = False, label: str = "") -> Superframe:
    """One superframe.  Give N (frame_bytes = 24 N) or frame_bytes.  starts: the n_aus-1 table entries, any 12-bit values
    (default: even split).  Corruptions made before the RS parity is computed, so RS cannot repair them: bad_crc (AU indices
    whose payload byte 0, or CRC byte 0 when the AU is empty, is flipped after its CRC) and bad_fire (fire code byte 0
    flipped).  Byte errors after the parity: Superframe.with_errors."""
    frame_bytes = frame_bytes or 24 * N
    total = 5 * frame_bytes
    N = total // 120
    n_aus = N_AUS[(dac_rate, sbr)]
    starts = even_starts(N, n_aus) if starts is None else list(starts)
    assert len(starts) == n_aus - 1 and all(0 <= s <= AU_START_MAX for s in starts)
    sf = np.zeros(total, dtype=np.uint8)
    sf[120 * N:] = rng.integers(0, 256, size=total - 120 * N, dtype=np.uint8)   # bytes after the last codeword
    sf[2] = (dac_rate << 6) | (sbr << 5) | (stereo << 4) | (ps << 3) | mpeg
    acc = 0
    for s in starts:
        acc = (acc << 12) | s
    nbits = 12 * len(starts)
    hdr = header_len(n_aus)
    if nbits:
        acc <<= (8 * (hdr - 3) - nbits)
        sf[3:hdr] = np.frombuffer(acc.to_bytes(hdr - 3, "big"), dtype=np.uint8)
    # the decoder's walk (aac_frame_processor.cpp:281-320): AU i = [bound[i], bound[i+1]), stop at the first one out of bounds
    bounds = [hdr] + starts + [110 * N]
    aus = []
    for i in range(n_aus):
        a, b = bounds[i], bounds[i + 1]
        if b - a - 2 < 0 or b >= total:
            break
        assert b <= 110 * N or a >= 120 * N, f"AU {i} [{a}, {b}) would overlap the RS parity"
        payload = rng.integers(0, 256, size=b - a - 2, dtype=np.uint8)
        crc = tx.crc16_ccitt(payload)
        sf[a:b - 2] = payload
        sf[b - 2], sf[b - 1] = crc >> 8, crc & 0xFF
        aus.append((a, b - a - 2))
    for i in bad_crc:
        sf[aus[i][0]] ^= 0x5A
    fc = tx.firecode(sf[2:11])
    sf[0], sf[1] = fc >> 8, fc & 0xFF
    if bad_fire:
        sf[0] ^= 0x01
    for i in range(N):
        sf[110 * N + i::N][:10] = np.array(tx.rs_encode(sf[i:110 * N:N].tolist(), 10), dtype=np.uint8)
    return Superframe(sf, frame_bytes, aus, label or f"starts {starts}", bad_crc, bad_fire)


def cw_errors(rng, cw: int, k: int, positions=None) -> list:
    """k byte errors in codeword cw at distinct random positions (or the given ones)"""
    pos = rng.choice(120, size=k, replace=False) if positions is None else positions
    return [(cw, int(p), int(rng.integers(1, 256))) for p in pos]


def event_log(events) -> bytes:
    """the flat observer log (oracle/ref_harness.cpp layout) of parsed events, what the GPU API returns"""
    out = b""
    for ev in events:
        out += np.array(ev[:5] + (len(ev[5]),), dtype=np.int32).tobytes() + ev[5] + b"\0" * ((-len(ev[5])) % 4)
    return out


def fit_lengths(N: int, n_aus: int, wanted) -> list:
    """payload lengths for AUs 0 .. n_aus-2 taken from `wanted` (cyclically), cut so that every AU fits in 110 N bytes"""
    room = 110 * N - header_len(n_aus) - 2 * n_aus
    lens = []
    for i in range(n_aus - 1):
        n = min(int(wanted[i % len(wanted)]), max(room, 0))
        lens.append(n)
        room -= n
    return lens


def program(tx, rng, N: int, dac_rate: int, sbr: int, mpeg: int = 0, rs_fails=None) -> list:
    """The superframes one processor is fed for size N and one AU layout, each meant to be decoded while synced: AU layouts
    (even, short and empty AUs, the longest AU the layout allows, AUs on both sides of 2115 bytes), AU CRC and fire-code
    failures, 0-5 byte errors per codeword anywhere (header, data, parity), uncorrectable codewords first, last and in a
    later pass of the decoder's 8 codewords, several in one pass, and AU-start tables the decoder must stop at.  Failing
    superframes are never more than four in a row, so the processor stays synced.  rs_fails(codeword) -> True when the RS
    decoder gives up on those 120 bytes: 6 or more errors usually make it give up, but the decoder searches the 135 padding
    positions too and sometimes finds a "correction" there, so uncorrectable error patterns are redrawn until it does."""
    n_aus = N_AUS[(dac_rate, sbr)]

    def bad(cw, k):
        while True:
            errs = cw_errors(rng, cw, k)
            cwb = base.sf[cw:120 * N:N].copy()
            for _, p, v in errs:
                cwb[p] ^= v
            if rs_fails is None or rs_fails(cwb):
                return errs

    hdr = header_len(n_aus)
    kw = dict(dac_rate=dac_rate, sbr=sbr, stereo=N & 1, ps=(N >> 1) & 1, mpeg=mpeg)
    out = []
    base = build(tx, rng, N, label="even split", **kw)
    out.append(base)
    out.append(build(tx, rng, N, starts=split_starts(N, n_aus, fit_lengths(N, n_aus, (0, 1, 31, 32, 33, 63))), label="AUs of 0, 1, 31, 32, 33, 63 bytes", **kw))
    out.append(build(tx, rng, N, starts=split_starts(N, n_aus, fit_lengths(N, n_aus, (63, 33, 0, 32, 1, 31)[::-1])), label="AUs of 31, 1, 32, 0, 33, 63 bytes", **kw))
    out.append(build(tx, rng, N, starts=split_starts(N, n_aus, [0] * (n_aus - 1)), label="longest last AU", **kw))
    for n in (2114, 2115, 2153):
        if hdr + n + 2 * n_aus <= 110 * N and hdr + n + 2 <= AU_START_MAX:
            out.append(build(tx, rng, N, starts=split_starts(N, n_aus, [n] + [0] * (n_aus - 2)), label=f"{n}-byte AU 0", **kw))
    out.append(build(tx, rng, N, bad_crc=(N % n_aus,), label=f"AU {N % n_aus} CRC", **kw))
    out.append(base.with_errors(sum((cw_errors(rng, cw, cw % 6) for cw in range(N)), []), "0-5 errors per codeword"))
    out.append(build(tx, rng, N, bad_crc=tuple(range(n_aus)), label="every AU CRC", **kw))
    five = cw_errors(rng, 0, 5, (0, 1, 2, 110, 119)) + (cw_errors(rng, N - 1, 5) if N > 1 else [])
    out.append(base.with_errors(five, "5 errors in codeword 0 (fire code, header, parity) and in codeword N-1"))
    out.append(base.with_errors(bad(N - 1, 6), "6 errors in codeword N-1", rs_fail=N - 1))
    out.append(base.with_errors(bad(0, 12) + cw_errors(rng, N - 1, 3), "12 errors in codeword 0", rs_fail=0))
    out.append(build(tx, rng, N, bad_fire=True, label="fire code", **kw))
    if N > 8:
        late = 8 + (N - 9) // 2
        errs = cw_errors(rng, 3, 5) + bad(late, 7) + cw_errors(rng, N - 1, 9)
        out.append(base.with_errors(errs, f"7 errors in codeword {late} (pass {late // 8})", rs_fail=late))
        out.append(base)
    if N >= 3:
        errs = cw_errors(rng, 0, 2) + bad(1, 6) + bad(2, 8)
        out.append(base.with_errors(errs, "codewords 1 and 2 uncorrectable", rs_fail=1))
    # AU-start tables the decoder stops at: start at / beyond the superframe end, decreasing, previous + 1; previous + 2 is an
    # empty AU and valid
    even = even_starts(N, n_aus)
    if n_aus > 1:
        j = n_aus - 2
        if 120 * N <= AU_START_MAX:
            out.append(build(tx, rng, N, starts=even[:j] + [120 * N], label=f"AU start {j + 1} at the superframe end", **kw))
            out.append(build(tx, rng, N, starts=even[:j] + [AU_START_MAX], label=f"AU start {j + 1} beyond the superframe end", **kw))
        prev = even[j - 1] if j else hdr
        out.append(build(tx, rng, N, starts=even[:j] + [prev - 1], label=f"AU start {j + 1} decreasing", **kw))
        out.append(build(tx, rng, N, starts=even[:j] + [prev + 1], label=f"AU start {j + 1} = previous + 1", **kw))
        out.append(build(tx, rng, N, starts=even[:j] + [prev + 2], label=f"AU start {j + 1} = previous + 2", **kw))
        out.append(build(tx, rng, N, starts=[hdr + 2] * (n_aus - 1) if n_aus > 2 else [hdr - 1], label="AU starts repeated", **kw))
    return out
