"""The C++ host side above the C ABI (sdrplusplus-dab-radio-plugin_b200/host/dab_adapters.hpp): classes with the
reference's names and signatures, driven by tests/host/adapter_check.cpp the way the reference's own code drives them,
compared with the oracle.  Bar: bit-exact for the integer half; soft bits within one quantisation step for OFDM.
"""
import importlib
import os
import struct
import subprocess
import tempfile

import numpy as np
import pytest

PKG = "sdrplusplus-dab-radio-plugin_b200"

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def driver(gpu_ctx):
    b = importlib.import_module(PKG + ".build")
    b.build()
    return b.build_adapter_check()


def _run(driver, what, payload: bytes) -> bytes:
    with tempfile.TemporaryDirectory() as d:
        fin, fout = os.path.join(d, "in.bin"), os.path.join(d, "out.bin")
        open(fin, "wb").write(payload)
        res = subprocess.run([driver, what, fin, fout], capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr
        return open(fout, "rb").read()


def _i32(*v):
    return struct.pack(f"<{len(v)}i", *v)


def _pi_code(tx, pi):
    if pi == 0:
        return np.array([1, 1, 0, 0] * 6, dtype=np.uint8)
    c = tx.pi_counts(pi)
    return np.array([1 if r < c[g] else 0 for g in range(8) for r in range(4)], dtype=np.uint8)


def test_dab_viterbi_decoder_class(driver, tx, pyref):
    """reset / update(punctured, code, n) x segments / chainback == DAB_Viterbi_Decoder, incl. a code outside table 13."""
    rng = np.random.default_rng(5)
    jobs = []
    for sg in (tx.FIC_SEGMENTS, tx.eep_segments(48, 2, False), tx.uep_segments(4), tx.eep_segments(54, 2, True)):
        n_in = int(tx.puncture_mask(sg).sum())
        info = rng.integers(0, 256, size=(sum(b for _, b in sg) // 4 - 6) // 8, dtype=np.uint8)
        soft = tx.hard_to_soft(tx.channel_encode(info, sg), rng, snr_db=2.0)
        assert soft.size == n_in
        jobs.append((sg, [(_pi_code(tx, pi), nb) for pi, nb in sg], soft))
    # an arbitrary 32-entry puncturing vector that is not a row of the table (de-punctured on the host, sent as PI_24)
    custom = np.array([1, 0, 1, 1] * 8, dtype=np.uint8)
    nbits = 128 * 6
    kept = sum(int(custom[i % 32]) for i in range(nbits))
    soft_c = rng.integers(-127, 128, size=kept + 12).astype(np.int8)
    jobs.append((None, [(custom, nbits), (_pi_code(tx, 0), 24)], soft_c))
    payload = _i32(len(jobs))
    for _, segs, soft in jobs:
        payload += _i32(len(segs))
        for code, nb in segs:
            payload += _i32(code.size) + code.tobytes() + _i32(nb)
        n_out = (sum(nb for _, nb in segs) // 4 - 6) // 8
        payload += _i32(soft.size) + soft.tobytes() + _i32(n_out)
    out = _run(driver, "viterbi", payload)
    port = pyref.PortViterbi()
    off = 0
    for sg, segs, soft in jobs:
        n_out = (sum(nb for _, nb in segs) // 4 - 6) // 8
        consumed, = struct.unpack_from("<i", out, off)
        err, = struct.unpack_from("<Q", out, off + 4)
        got = np.frombuffer(out, dtype=np.uint8, count=n_out, offset=off + 12)
        off += 12 + n_out
        if sg is not None:
            exp, exp_consumed, exp_err = port.decode(soft, sg)
            assert consumed == exp_consumed and err == exp_err
            assert np.array_equal(got, exp)
        else:
            # expectation: de-puncture by hand, decode as the unpunctured mother code
            full, j = [], 0
            for code, nb in segs:
                for i in range(nb):
                    if code[i % code.size]:
                        full.append(int(soft[j])); j += 1
                    else:
                        full.append(0)
            exp, _, exp_err = port.decode(np.array(full, dtype=np.int8), [(24, len(full))])
            assert consumed == j and err == exp_err
            assert np.array_equal(got, exp[:n_out])


def test_fic_decoder_class(driver, tx, pyref):
    rng = np.random.default_rng(6)
    ens = tx.EnsembleTx(1, tx.default_ensemble(), seed=3)
    frame = ens.next_frame_bits()
    groups = [tx.hard_to_soft(frame[c * 2304:(c + 1) * 2304], rng, snr_db=snr) for c, snr in zip(range(4), (8.0, 2.0, -2.0, -8.0))]
    out = _run(driver, "fic", _i32(4) + b"".join(g.tobytes() for g in groups))
    o = pyref.RefFic() if pyref.ref_available() else pyref.PortFic()
    off = 0
    total = 0
    for c, g in enumerate(groups):
        n, = struct.unpack_from("<i", out, off)
        fibs = [out[off + 4 + 30 * i: off + 4 + 30 * (i + 1)] for i in range(n)]
        off += 4 + 30 * n
        assert fibs == o.decode_group(g, c)
        total += n
    assert total >= 6   # the clean groups deliver their FIBs, the noisy ones fail the CRC and stay silent


@pytest.mark.parametrize("sub", ["eep3a", "uep", "eep2b"])
def test_msc_decoder_class(driver, tx, pyref, sub):
    sc = {"eep3a": tx.Subchannel(0, 12, 48, eep_level=2), "uep": tx.Subchannel(1, 100, 35, is_uep=True, uep_index=4, dabplus=False),
          "eep2b": tx.Subchannel(2, 300, 42, eep_level=1, eep_type_b=True, dabplus=False)}[sub]
    ens = tx.EnsembleTx(1, [sc], seed=21)
    rng = np.random.default_rng(8)
    cifs = []
    for _ in range(6):
        f = ens.next_frame_bits()
        for c in range(4):
            cifs.append(tx.hard_to_soft(f[9216 + c * 55296: 9216 + (c + 1) * 55296], rng, snr_db=4.0))
    payload = _i32(0, sc.start_address, sc.length, int(sc.is_uep), sc.uep_index, sc.eep_level,
                   int(sc.eep_type_b), 0, len(cifs)) + b"".join(c.tobytes() for c in cifs)
    out = _run(driver, "msc", payload)
    mk = pyref.RefMsc if pyref.ref_available() else pyref.PortMsc
    o = mk(sc.start_address, sc.length, sc.is_uep, sc.uep_index, sc.eep_level, sc.eep_type_b)
    off = 0
    n_valid = 0
    for c in cifs:
        n, = struct.unpack_from("<i", out, off)
        got = np.frombuffer(out, dtype=np.uint8, count=n, offset=off + 4)
        off += 4 + n
        exp = o.decode_cif(c)
        assert n == exp.size
        assert np.array_equal(got, exp)
        n_valid += int(n > 0)
    assert n_valid == len(cifs) - 15   # the first 15 CIFs only fill the time de-interleaver


def test_reed_solomon_decoder_class(driver, tx, pyref):
    rng = np.random.default_rng(9)
    cws = []
    for n_err in (0, 1, 3, 5, 6, 9):
        data = rng.integers(0, 256, size=110, dtype=np.uint8)
        cw = np.array(list(data) + tx.rs_encode(list(data)), dtype=np.uint8)
        pos = rng.choice(120, size=n_err, replace=False)
        cw[pos] ^= rng.integers(1, 256, size=n_err).astype(np.uint8)
        cws.append(cw)
    out = _run(driver, "rs", _i32(len(cws), 10, 135) + b"".join(c.tobytes() for c in cws))
    o = pyref.RefRS() if pyref.ref_available() else pyref.PortRS()
    off = 0
    for cw in cws:
        cnt, = struct.unpack_from("<i", out, off)
        got = np.frombuffer(out, dtype=np.uint8, count=120, offset=off + 4)
        pos = np.frombuffer(out, dtype=np.int32, count=10, offset=off + 124)
        off += 4 + 120 + 40
        e_cnt, e_data, e_pos = o.decode(cw)
        assert cnt == e_cnt
        assert np.array_equal(got, e_data)
        if cnt > 0:
            assert np.array_equal(pos[:cnt], np.asarray(e_pos)[:cnt])


def test_aac_frame_processor_class(driver, tx, pyref):
    """Superframe sync, RS correction, fire code and AU CRC events fire in the reference's order with the same payloads."""
    rng = np.random.default_rng(10)
    frames = []
    frames += [rng.integers(0, 256, size=192, dtype=np.uint8) for _ in range(3)]      # garbage before the first superframe
    for k in range(4):
        sf = np.array(tx.build_superframe(64, rng), dtype=np.uint8).copy()
        if k == 1:
            sf[rng.choice(sf.size, size=12, replace=False)] ^= 0x5A                  # correctable byte errors
        if k == 2:
            sf[200:260] ^= 0xFF                                                       # burst: some codewords uncorrectable
        frames += [sf[i * 192:(i + 1) * 192] for i in range(5)]
    out = _run(driver, "aac", _i32(len(frames), 192) + b"".join(f.tobytes() for f in frames))
    o = pyref.RefAac() if pyref.ref_available() else pyref.PortAac()
    off = 0
    seen = set()
    for f in frames:
        n, = struct.unpack_from("<i", out, off)
        off += 4
        got = []
        for _ in range(n):
            t, a, b, c, d, ln = struct.unpack_from("<6i", out, off)
            got.append((t, a, b, c, d, bytes(out[off + 24: off + 24 + ln])))
            off += 24 + ln
            seen.add(t)
        assert got == o.process(f)
    assert {pyref.EV_HEADER, pyref.EV_AU}.issubset(seen)


def test_radio_block_chain(driver, tx, pyref):
    """Radio_Block: complex<float> blocks into OFDM_Demod::Process, soft bits stay on the device, FIBs and sub-channel bytes
    come out of the BasicRadio observers.  The frames and soft bits match the reference OFDM_Demod on the same recording (one LSB);
    the FIBs and bytes equal the reference's FIC and MSC decoders fed the frames the adapter emitted and, where the reference build
    is the oracle, fed the reference's own frames."""
    mode, block = 1, 65536
    subs = [tx.Subchannel(0, 0, 48, eep_level=2), tx.Subchannel(1, 48, 54, eep_level=2, eep_type_b=True, dabplus=False)]
    ens = tx.EnsembleTx(mode, subs, seed=77)
    n_frames = 7
    iq = tx.ofdm_modulate([ens.next_frame_bits() for _ in range(n_frames)], mode)
    u8 = tx.to_u8(tx.impair(iq, 16.0, 2.2e-3, 4321, seed=5, tail_samples=3000), 30.0)
    n = (u8.size // 2 // block) * block
    payload = _i32(mode, len(subs))
    for sc in subs:
        payload += _i32(0, sc.start_address, sc.length, int(sc.is_uep), sc.uep_index, sc.eep_level, int(sc.eep_type_b), int(sc.dabplus))
    payload += _i32(block, n) + u8[:2 * n].tobytes()
    out = _run(driver, "radio", payload)

    use_ref = pyref.ref_available()
    o = pyref.RefOfdm(mode, 1) if use_ref else pyref.PortOfdm(mode)
    c32 = ((u8[:2 * n].astype(np.float32) - np.float32(127.5)) * np.float32(1.0 / 127.5)).view(np.complex64)
    for off in range(0, n, block):
        o.process_c32(c32[off:off + block])
    exp_frames = o.pop_frames()

    def decode(soft_frames):
        """FIBs and per-sub-channel bytes of the oracle's FIC and MSC decoders over these soft-bit frames"""
        o_fic = pyref.RefFic() if use_ref else pyref.PortFic()
        mk = pyref.RefMsc if use_ref else pyref.PortMsc
        o_msc = [mk(sc.start_address, sc.length, sc.is_uep, sc.uep_index, sc.eep_level, sc.eep_type_b) for sc in subs]
        exp_fibs, exp_msc = [], [[] for _ in subs]
        for b in soft_frames:
            for c in range(4):
                exp_fibs += o_fic.decode_group(b[c * 2304:(c + 1) * 2304], c)
            for k in range(len(subs)):
                for c in range(4):
                    e = o_msc[k].decode_cif(b[9216 + c * 55296:9216 + (c + 1) * 55296])
                    if e.size:
                        exp_msc[k].append(e)
        return exp_fibs, exp_msc

    # the reference order per frame would be FIBs then sub-channels (BasicRadio::Process); the adapter decodes the frame
    # on the device first and then reports the soft bits, so the records are grouped by tag before comparing
    off = 0
    frames, fibs, msc = [], [], [[] for _ in subs]
    while True:
        tag, = struct.unpack_from("<i", out, off)
        off += 4
        if tag == 0:
            total_read, total_desync, state = struct.unpack_from("<3i", out, off)
            break
        if tag == 1:
            ln, = struct.unpack_from("<i", out, off)
            bits = np.frombuffer(out, dtype=np.int8, count=ln, offset=off + 4)
            fto, = struct.unpack_from("<i", out, off + 4 + ln)
            frames.append((bits, fto))
            off += 8 + ln
        elif tag == 2:
            fibs.append(out[off:off + 30])
            off += 30
        else:
            k, ln = struct.unpack_from("<2i", out, off)
            msc[k].append(np.frombuffer(out, dtype=np.uint8, count=ln, offset=off + 8))
            off += 8 + ln
    assert len(frames) == len(exp_frames) >= n_frames - 2
    assert total_read == len(exp_frames)
    for (bits, fto), (eb, _, _, et) in zip(frames, exp_frames):
        assert fto == et
        assert np.abs(bits.astype(np.int32) - eb.astype(np.int32)).max() <= 1
    # one LSB can flip a Viterbi decision, so the exact comparison feeds the oracle's decoders the soft bits the adapter reported
    # (the ones it decoded).  The C restatement's OFDM is itself only within one LSB of the reference's, so the end-to-end
    # comparison with the oracle's own frames is made where the reference build is the oracle.
    sources = [[b for b, _ in frames]] + ([[e[0] for e in exp_frames]] if use_ref else [])
    for src in sources:
        exp_fibs, exp_msc = decode(src)
        assert fibs == exp_fibs
        for k in range(len(subs)):
            assert len(msc[k]) == len(exp_msc[k])
            for a, b in zip(msc[k], exp_msc[k]):
                assert np.array_equal(a, b)


def test_basic_radio_configures_itself_from_the_fic(driver, tx, pyref):
    """BasicRadio with EnableSelfConfiguration(): soft-bit frames in, channels announced through On_Audio_Channel as the FIC
    completes them (FIG 0/1 + 0/2), then their bytes equal the oracle's MSC decoders started at the same frame."""
    rng = np.random.default_rng(8)
    subs = [tx.Subchannel(5, 0, 48, eep_level=2), tx.Subchannel(11, 48, 54, eep_level=2, eep_type_b=True, dabplus=False),
            tx.Subchannel(20, 102, 35, is_uep=True, uep_index=4, dabplus=False)]
    ens = tx.EnsembleTx(1, subs, seed=31)
    n_frames = 9
    frames = [tx.hard_to_soft(ens.next_frame_bits(), rng, snr_db=7.0) for _ in range(n_frames)]
    out = _run(driver, "selfcfg", _i32(1, n_frames, frames[0].size) + b"".join(f.tobytes() for f in frames))
    announced, data, off = [], {}, 0
    while True:
        tag, = struct.unpack_from("<i", out, off)
        off += 4
        if tag == 0:
            n_channels, = struct.unpack_from("<i", out, off)
            break
        if tag == 4:
            announced.append(struct.unpack_from("<9i", out, off))
            off += 36
        else:
            sid, ln = struct.unpack_from("<2i", out, off)
            data.setdefault(sid, []).append(np.frombuffer(out, dtype=np.uint8, count=ln, offset=off + 8))
            off += 8 + ln
    assert n_channels == len(subs)
    assert [a[0] for a in announced] == [s.id for s in subs]
    for a, s in zip(announced, subs):
        assert a[1:4] == (s.start_address, s.length, int(s.is_uep)) and a[7] == int(s.dabplus) and a[8] == 0   # all known after the first frame
        assert (a[4] == s.uep_index) if s.is_uep else (a[5:7] == (s.eep_level, int(s.eep_type_b)))
    mk = pyref.RefMsc if pyref.ref_available() else pyref.PortMsc
    for s in subs:
        o = mk(s.start_address, s.length, s.is_uep, s.uep_index, s.eep_level, s.eep_type_b)
        exp = []
        for f in frames[1:]:                      # the decoder exists from the frame after the one that configured it
            for c in range(4):
                e = o.decode_cif(f[9216 + c * 55296: 9216 + (c + 1) * 55296])
                if e.size:
                    exp.append(e)
        got = data.get(s.id, [])
        assert len(got) == len(exp) > 0, s.id
        assert all(np.array_equal(g, e) for g, e in zip(got, exp)), s.id


def test_msc_decoder_objects_share_a_pool_context(driver, tx, pyref):
    """Three MSC_Decoder objects alive at once (one leased stream each of a shared pool context), fed interleaved: each equals its
    own oracle decoder.  The first one re-uses a stream that another decoder held before: it must start empty."""
    scs = [tx.Subchannel(0, 12, 48, eep_level=2), tx.Subchannel(1, 100, 35, is_uep=True, uep_index=4, dabplus=False),
           tx.Subchannel(2, 300, 42, eep_level=1, eep_type_b=True, dabplus=False)]
    rng = np.random.default_rng(18)
    n_cifs = 20
    cifs = [[rng.integers(-127, 128, size=55296).astype(np.int8) for _ in scs] for _ in range(n_cifs)]
    payload = _i32(len(scs))
    for sc in scs:
        payload += _i32(sc.id, sc.start_address, sc.length, int(sc.is_uep), sc.uep_index, sc.eep_level, int(sc.eep_type_b), 0)
    payload += _i32(n_cifs) + b"".join(c.tobytes() for row in cifs for c in row)
    out = _run(driver, "mscpool", payload)
    mk = pyref.RefMsc if pyref.ref_available() else pyref.PortMsc
    o = [mk(sc.start_address, sc.length, sc.is_uep, sc.uep_index, sc.eep_level, sc.eep_type_b) for sc in scs]
    off, n_valid = 0, 0
    for row in cifs:
        for k, c in enumerate(row):
            n, = struct.unpack_from("<i", out, off)
            got = np.frombuffer(out, dtype=np.uint8, count=n, offset=off + 4)
            off += 4 + n
            exp = o[k].decode_cif(c)
            assert n == exp.size and np.array_equal(got, exp), k
            n_valid += int(n > 0)
    assert n_valid == len(scs) * (n_cifs - 15)


def test_ofdm_demod_class_serves_the_gui_getters(driver, tx, pyref, ref_ok):
    """OFDM_Demod::GetImpulseResponse / GetCoarseFrequencyResponse / GetFrameFFT / GetFrameDataVec / GetCorrelationTimeBuffer
    (ofdm_demodulator.h:135-140, read by src/render_radio_block.cpp:96-214) through the C++ adapter: the reference's extents,
    contents within the tolerances of tests/test_ofdm_gpu.py::test_gui_taps_match_reference."""
    mode, block = 1, 65536
    ens = tx.EnsembleTx(mode, tx.default_ensemble(), seed=5)
    iq = tx.ofdm_modulate([ens.next_frame_bits() for _ in range(4)], mode)
    u8 = tx.to_u8(tx.impair(iq, 18.0, 1.7e-3, 2222, seed=6, tail_samples=3000), 30.0)
    n = (u8.size // 2 // block) * block
    out = _run(driver, "taps", _i32(mode, block, n) + u8[:2 * n].tobytes())
    ref = pyref.RefOfdm(mode, 1)
    c32 = ((u8[:2 * n].astype(np.float32) - np.float32(127.5)) * np.float32(1.0 / 127.5)).view(np.complex64)
    for off in range(0, n, block):
        ref.process_c32(c32[off:off + block])
    P = importlib.import_module(PKG).get_params(mode)
    N, L, K = P.nb_fft, P.nb_frame_symbols, P.nb_data_carriers
    off = 0
    frames, = struct.unpack_from("<i", out, off); off += 4
    assert frames == len(ref.pop_frames()) >= 2

    def take(dtype, per):
        nonlocal off
        cnt, = struct.unpack_from("<i", out, off)
        a = np.frombuffer(out, dtype=dtype, count=cnt, offset=off + 4)
        off += 4 + cnt * per
        return a

    imp, coarse = take(np.float32, 4), take(np.float32, 4)
    fft, vec, corr = take(np.complex64, 8), take(np.complex64, 8), take(np.complex64, 8)
    assert imp.size == N and coarse.size == N and fft.size == (L + 1) * N and vec.size == (L - 1) * N and corr.size == P.nb_null_period + P.nb_symbol_period
    for got, exp in ((imp, ref.impulse_response(N)), (coarse, ref.coarse_response(N))):
        assert int(np.argmax(got)) == int(np.argmax(exp))
        strong = exp > exp.max() - 40.0
        assert np.abs(got[strong] - exp[strong]).max() < 0.05
    exp_fft = ref.frame_fft((L + 1) * N)
    scale = np.abs(exp_fft).max()
    assert np.abs(fft - exp_fft).max() < 2e-3 * scale
    exp_vec = ref.frame_data_vec((L - 1) * K)
    assert np.abs(vec[:(L - 1) * K] - exp_vec).max() < 4e-3 * np.abs(exp_vec).max()
    assert np.array_equal(corr, ref.correlation_buffer(corr.size))   # raw input samples: identical


def test_ofdm_demod_config_edits_between_process_calls(driver, pyref):
    """OFDM_Demod::GetConfig() edited between Process() calls of varying lengths, every field at once (host/dab_adapters.hpp
    push_config copies them into dabgpu_ofdm_config one by one): after each call the frames and GetState / GetTotalFramesRead /
    GetTotalFramesDesync / GetFineTimeOffset / GetSignalAverage / GetCoarseFrequencyOffset / GetFineFrequencyOffset are the
    oracle's under the same edits.  The edits are those of tests/ofdm_config_cases.py, which tests/test_ofdm_config_cpu.py shows
    change the oracle's output whenever two fields of the same type are exchanged."""
    import ofdm_config_cases as C
    mode = C.ADAPTER_MODE
    use_ref = pyref.ref_available()
    recs = C.recordings(mode)
    n = recs.shape[1] // 2
    cl = C.partition_calls(n, C.ADAPTER_BLOCKS)
    frame_bits = importlib.import_module(PKG).get_params(mode).nb_frame_bits
    for s in C.ADAPTER_STREAMS:
        u8 = recs[s]
        payload = _i32(mode, len(C.ADAPTER_EDITS))
        for k, e in sorted(C.ADAPTER_EDITS.items()):
            payload += _i32(k) + struct.pack("<8f", *[e[f] for f in C.FLOAT_KNOBS]) + _i32(*[e[f] for f in C.INT_KNOBS])
        payload += _i32(len(cl), *[ln for _, ln in cl]) + u8[:2 * n].tobytes()
        out = _run(driver, "ofdmcfg", payload)
        exp = C.oracle_outputs(pyref, mode, C.to_c32(u8[None, :2 * n]), {}, cl, 0, u8=False, use_ref=use_ref, edits=C.ADAPTER_EDITS)[0]
        off, frames = 0, []
        for k in range(len(cl)):
            nf, = struct.unpack_from("<i", out, off)
            off += 4
            for _ in range(nf):
                bits = np.frombuffer(out, dtype=np.int8, count=frame_bits, offset=off)
                coarse, fine, fto = struct.unpack_from("<2fi", out, off + frame_bits)
                frames.append((bits, coarse, fine, fto))
                off += frame_bits + 12
            state, read, desync, fto = struct.unpack_from("<4i", out, off)
            l1, coarse, fine = struct.unpack_from("<3f", out, off + 16)
            off += 28
            e = exp["status"][k]
            tag = f"stream {s} after call {k}"
            assert (state, read, desync, fto) == (e["state"], e["frames_read"], e["frames_desync"], e["fine_time_offset"]), (tag, e)
            assert abs(l1 - e["signal_avg"]) <= C.L1_RTOL * abs(e["signal_avg"]), (tag, l1, e)
            assert abs(coarse - e["coarse"]) <= C.FREQ_ATOL and abs(fine - e["fine"]) <= C.FREQ_ATOL, (tag, coarse, fine, e)
        assert off == len(out)
        assert len(frames) == len(exp["frames"]) > 0
        for i, ((gb, gc, gf, gt), (eb, ec, ef, et)) in enumerate(zip(frames, exp["frames"])):
            assert gt == et and abs(gc - ec) <= C.FREQ_ATOL and abs(gf - ef) <= C.FREQ_ATOL, (s, i)
            d = np.abs(gb.astype(np.int32) - eb.astype(np.int32))
            if (d >= 1).mean() < 1e-3:
                assert d.max() <= 1, (s, i, d.max())
            else:
                assert d.max() <= 16 and (d > 1).mean() <= 5e-4, (s, i, d.max())
