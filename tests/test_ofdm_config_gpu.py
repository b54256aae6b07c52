"""The OFDM control kernel under every synchronisation knob set (dabgpu_ofdm_config = OFDM_Demod_Config), under knob changes
between Process() calls, and under arbitrary Process() partitions, against the oracle (the reference build where present, else
the C restatement), in every transmission mode.  tests/test_ofdm_config_cpu.py shows that each case changes the oracle's output,
so a build that ignored a knob, a change or the partition fails here.

After every call and for every stream: state, frame and desync counts and fine time offset equal, signal_l1_average within 1e-5
relative, coarse and fine frequency within 2e-6.  Every frame: same count and fine time offset, coarse and fine within 2e-6, soft
bits by the rule of tests/test_robustness_full_gpu.py.
"""
import functools

import numpy as np
import pytest

import ofdm_config_cases as C

pytestmark = pytest.mark.gpu

SOFT_TOL, SOFT_TOL_WEAK, WEAK_FRACTION = 1, 16, 5e-4   # tests/test_robustness_full_gpu.py


@functools.lru_cache(maxsize=None)
def _recordings(mode):
    return C.recordings(mode)


def _input(mode, u8):
    iq = _recordings(mode)
    return iq if u8 else C.to_c32(iq)


def _oracle(pyref, mode, iq, cfg, cl, bs, u8=True, edits=None):
    return C.oracle_outputs(pyref, mode, iq, cfg, cl, bs, u8=u8, use_ref=pyref.ref_available(), edits=edits)


def _gpu_run(g, iq, cl, bs, u8=True, edits=None):
    """dabgpu_ofdm_process per call, knob edits before the calls that have one; status and frames of every stream after each call"""
    out = [{"status": [], "frames": []} for _ in range(iq.shape[0])]
    for k, (off, ln) in enumerate(cl):
        if edits and k in edits:
            g.ofdm_set_config(**edits[k])
        g.ofdm_process(iq[:, 2 * off:2 * (off + ln)] if u8 else iq[:, off:off + ln], block_size=bs)
        for s, r in enumerate(out):
            r["status"].append(g.ofdm_status(s))
            r["frames"] += g.ofdm_pop_frames(s)
    return out


def _assert_soft(got, exp, tag):
    d = np.abs(got.astype(np.int32) - exp.astype(np.int32))
    if (d >= 1).mean() < 1e-3:
        assert d.max() <= SOFT_TOL, f"{tag}: max soft-bit delta {d.max()}"
    else:
        assert d.max() <= SOFT_TOL_WEAK and (d > SOFT_TOL).mean() <= WEAK_FRACTION, \
            f"{tag}: max soft-bit delta {d.max()}, {(d > SOFT_TOL).sum()} bits beyond one step"


def _assert_status(a, b, tag):
    assert (a["state"], a["total_frames_read"], a["total_frames_desync"], a["fine_time_offset"]) == \
        (b["state"], b["frames_read"], b["frames_desync"], b["fine_time_offset"]), (tag, a, b)
    assert abs(a["signal_l1_average"] - b["signal_avg"]) <= C.L1_RTOL * abs(b["signal_avg"]), (tag, a, b)
    assert abs(a["freq_coarse_offset"] - b["coarse"]) <= C.FREQ_ATOL and abs(a["freq_fine_offset"] - b["fine"]) <= C.FREQ_ATOL, (tag, a, b)


def _assert_match(got, exp, tag, streams=None):
    for s, (g, e) in enumerate(zip(got, exp)):
        t = f"{tag} stream {s} {C.STREAMS[s] if streams is None else streams[s]}"
        assert len(g["status"]) == len(e["status"])
        for k, (a, b) in enumerate(zip(g["status"], e["status"])):
            _assert_status(a, b, f"{t} after call {k}")
        assert len(g["frames"]) == len(e["frames"]), t
        for i, ((gb, gc, gf, gt), (eb, ec, ef, et)) in enumerate(zip(g["frames"], e["frames"])):
            assert gt == et, f"{t} frame {i}: fine time offset {gt} != {et}"
            assert abs(gc - ec) <= C.FREQ_ATOL and abs(gf - ef) <= C.FREQ_ATOL, (t, i, gc, ec, gf, ef)
            _assert_soft(gb, eb, f"{t} frame {i}")


def _assert_identical(a, b, tag):
    for s, (x, y) in enumerate(zip(a, b)):
        assert x["status"] == y["status"], (tag, s)
        assert len(x["frames"]) == len(y["frames"]), (tag, s)
        for fx, fy in zip(x["frames"], y["frames"]):
            assert np.array_equal(fx[0], fy[0]) and fx[1:] == fy[1:], (tag, s)


KNOB_CASES = [(m, k, "u8") for m in (1, 2, 3, 4) for k in C.knob_cases(m)] + \
             [(m, k, "c32") for m in (1, 2, 3, 4) for k in C.knob_cases(m, c32=True)]


@pytest.mark.parametrize("mode,knob,fmt", KNOB_CASES, ids=[f"mode{m}-{k}-{f}" for m, k, f in KNOB_CASES])
def test_knob_set_matches_oracle(gpu_ctx, pyref, mode, knob, fmt):
    u8 = fmt == "u8"
    iq = _input(mode, u8)
    n = iq.shape[1] // 2 if u8 else iq.shape[1]
    cfg = C.case_config(knob, mode)
    cl = C.calls(n)
    g = gpu_ctx.DabGpu(mode=mode, max_streams=iq.shape[0], iq_format=gpu_ctx.IQ_U8 if u8 else gpu_ctx.IQ_C32)
    g.ofdm_set_config(**cfg)                   # = ofdm_overrides at creation (test_config_at_creation_equals_set_config)
    got = _gpu_run(g, iq, cl, C.CALL, u8)
    g.close()
    _assert_match(got, _oracle(pyref, mode, iq, cfg, cl, C.CALL, u8), f"mode {mode} {knob} {fmt}")


@pytest.mark.parametrize("mode", [1, 2, 3, 4])
def test_config_at_creation_equals_set_config(gpu_ctx, pyref, mode):
    """DabGpu(ofdm_overrides=cfg) (dabgpu_config.ofdm) and dabgpu_ofdm_set_config(cfg) before the first call: bit-identical, and
    both the oracle's"""
    iq = _input(mode, True)
    cfg = {**C.case_config("slow_beta_0.02", mode), **C.knobs("l1_37x1", mode), "fine_freq_update_beta": 0.7}
    cl = C.calls(iq.shape[1] // 2)
    g1 = gpu_ctx.DabGpu(mode=mode, max_streams=iq.shape[0], ofdm_overrides=cfg)
    g2 = gpu_ctx.DabGpu(mode=mode, max_streams=iq.shape[0])
    g2.ofdm_set_config(**cfg)
    a, b = _gpu_run(g1, iq, cl, C.CALL), _gpu_run(g2, iq, cl, C.CALL)
    g1.close()
    g2.close()
    _assert_identical(a, b, f"mode {mode}")
    _assert_match(a, _oracle(pyref, mode, iq, cfg, cl, C.CALL), f"mode {mode} at creation")


LIVE = ["null_search", "mid_frame", "after_desync", "coarse_toggle"]


@pytest.mark.parametrize("mode", [1, 2, 3, 4])
@pytest.mark.parametrize("scenario", LIVE)
def test_live_change_matches_oracle(gpu_ctx, pyref, mode, scenario):
    """dabgpu_ofdm_set_config between calls takes effect from the next call on, for every stream of the context; the oracle gets
    the same change at the same call boundary"""
    iq = _input(mode, True)
    cl = C.live_calls(iq.shape[1] // 2)
    cfg = C.LIVE_BASE[mode]
    edits = C.live_scenarios(mode, _oracle(pyref, mode, iq, cfg, cl, 0))[scenario]
    g = gpu_ctx.DabGpu(mode=mode, max_streams=iq.shape[0], ofdm_overrides=cfg)
    got = _gpu_run(g, iq, cl, 0, edits=edits)
    g.close()
    _assert_match(got, _oracle(pyref, mode, iq, cfg, cl, 0, edits=edits), f"mode {mode} {scenario} at calls {sorted(edits)}")


PARTITION_CASES = [(m, p, k, "u8") for m in (1, 2, 3, 4) for p, k in C.partition_cases(m)] + \
                  [(m, p, k, "c32") for m in (1, 2, 3, 4) for p, k in C.partition_cases(m, c32=True)]


@pytest.mark.parametrize("mode,part,knob,fmt", PARTITION_CASES, ids=[f"mode{m}-{p}-{k or 'base'}-{f}" for m, p, k, f in PARTITION_CASES])
def test_partition_matches_oracle(gpu_ctx, pyref, mode, part, knob, fmt):
    """Process() blocks of any size, calls that are not a multiple of the block size, ragged calls of one block each, in the
    smallest IQ ring that holds a block, so that L1 windows and frames straddle the ring's wrap"""
    u8 = fmt == "u8"
    iq = _input(mode, u8)
    n = iq.shape[1] // 2 if u8 else iq.shape[1]
    lengths, bs, limit = C.partitions(mode)[part]
    cfg = C.BASE[mode] if knob is None else C.case_config(knob, mode)
    cl = C.partition_calls(n, lengths, limit)
    ring = C.ring_for_block(mode, bs or max(lengths))
    g = gpu_ctx.DabGpu(mode=mode, max_streams=iq.shape[0], iq_format=gpu_ctx.IQ_U8 if u8 else gpu_ctx.IQ_C32, ring_samples=ring,
                       ofdm_overrides=cfg)
    got = _gpu_run(g, iq, cl, bs, u8)
    g.close()
    _assert_match(got, _oracle(pyref, mode, iq, cfg, cl, bs, u8), f"mode {mode} {part} {knob} {fmt} ring {ring}")


@pytest.mark.parametrize("mode", [1, 2, 3, 4])
def test_device_input_of_any_capacity_with_ragged_blocks(gpu_ctx, pyref, mode):
    """dabgpu_ofdm_attach_device_input with a capacity that is not a power of two (no wrap), fed by dabgpu_ofdm_advance in ragged
    calls of one block each"""
    import torch
    iq = _input(mode, True)
    S, n = iq.shape[0], iq.shape[1] // 2
    cap = n + 1001
    dev = torch.zeros((S, 2 * cap), dtype=torch.uint8, device="cuda:0")
    dev[:, :2 * n] = torch.from_numpy(iq).to("cuda:0")
    torch.cuda.synchronize()
    lengths, _, _ = C.partitions(mode)["ragged_calls"]
    cl = C.partition_calls(n, lengths)
    cfg = C.case_config(C.PARTITION_KNOBS, mode)
    g = gpu_ctx.DabGpu(mode=mode, max_streams=S, ofdm_overrides=cfg)
    g.ofdm_attach_device_input(dev.data_ptr(), cap, cap)
    got = [{"status": [], "frames": []} for _ in range(S)]
    for off, ln in cl:
        g.ofdm_advance(ln, block_size=0)
        for s, r in enumerate(got):
            r["status"].append(g.ofdm_status(s))
            r["frames"] += g.ofdm_pop_frames(s)
    g.close()
    del dev
    _assert_match(got, _oracle(pyref, mode, iq, cfg, cl, 0), f"mode {mode} device input capacity {cap}")


@pytest.mark.parametrize("mode", [1, 2, 3, 4])
def test_set_config_between_pipelined_submits(gpu_ctx, pyref, mode):
    """dabgpu_set_config between dabgpu_submit(t) and dabgpu_submit(t + 1) while earlier tickets are in flight acts exactly like
    the same change between dabgpu_ofdm_process calls t and t + 1: every launch takes the knobs by value when it is queued"""
    iq = _input(mode, True)
    S, n = iq.shape[0], iq.shape[1] // 2
    cl = C.calls(n)
    cfg = C.BASE[mode]
    edits = {3: dict(fine_freq_update_beta=0.3, signal_l1_nb_samples=37, signal_l1_nb_decimate=1),
             7: dict(coarse_freq_slow_beta=0.02, impulse_peak_threshold_db=15.0)}
    late = {k + 1: v for k, v in edits.items()}
    exp = _oracle(pyref, mode, iq, cfg, cl, C.CALL, edits=edits)
    assert C.differs(exp, _oracle(pyref, mode, iq, cfg, cl, C.CALL, edits=late)), "a change one call late would go unnoticed"

    g_sync = gpu_ctx.DabGpu(mode=mode, max_streams=S, ofdm_overrides=cfg)
    sync = _gpu_run(g_sync, iq, cl, C.CALL, edits=edits)
    _assert_match(sync, exp, f"mode {mode} synchronous")

    g = gpu_ctx.DabGpu(mode=mode, max_streams=S, ofdm_overrides=cfg)
    hb = gpu_ctx.HostBuffer(iq.nbytes)
    hb.array[:] = iq.reshape(-1)
    tickets = []
    for k, (off, ln) in enumerate(cl):
        if k in edits:
            g.ofdm_set_config(**edits[k])      # ticket k - 1 (and k - 2) still in flight
        tickets.append(g.submit(hb.ptr.value + 2 * off, 2 * n, ln, block_size=C.CALL))
        if len(tickets) >= 2:
            g.wait(tickets[-2])
    g.wait(tickets[-1])
    keys = ("state", "total_frames_read", "total_frames_desync", "fine_time_offset", "signal_l1_average", "freq_coarse_offset",
            "freq_fine_offset")
    for s in range(S):
        st = g.ofdm_status(s)
        assert [st[k] for k in keys] == [sync[s]["status"][-1][k] for k in keys], (mode, s)
        frames = g.ofdm_pop_frames(s)
        assert len(frames) == len(sync[s]["frames"]), (mode, s)
        for a, b in zip(frames, sync[s]["frames"]):
            assert np.array_equal(a[0], b[0]) and a[1:] == b[1:], (mode, s)
    g.close()
    g_sync.close()
    hb.close()


@pytest.mark.parametrize("mode", [1, 2, 3, 4])
def test_invalid_knobs_are_refused_and_keep_the_previous_ones(gpu_ctx, pyref, mode):
    """dabgpu_ofdm_set_config with a signal_l1 window of 0 or -1 returns DABGPU_ERR_INVALID, launches nothing and leaves the
    knobs in force: the calls after it still match the oracle under the old knobs.  dabgpu_ctx_create refuses the same."""
    iq = _input(mode, True)
    S, n = iq.shape[0], iq.shape[1] // 2
    cl = C.calls(n)
    cfg = C.case_config(C.PARTITION_KNOBS, mode)
    g = gpu_ctx.DabGpu(mode=mode, max_streams=S, ofdm_overrides=cfg)
    half = len(cl) // 2
    got = _gpu_run(g, iq, cl[:half], C.CALL)
    launches = g.launch_count
    for bad in (dict(signal_l1_nb_samples=0), dict(signal_l1_nb_samples=-1), dict(signal_l1_nb_decimate=0),
                dict(signal_l1_nb_decimate=-1), dict(signal_l1_nb_samples=0, signal_l1_nb_decimate=0)):
        with pytest.raises(gpu_ctx.DabGpuError) as e:
            g.ofdm_set_config(**bad)
        assert e.value.code == gpu_ctx.ERR_INVALID
    assert g.launch_count == launches
    g.ofdm_set_config()                        # re-applies the knobs the binding holds: the valid ones
    rest = _gpu_run(g, iq, [(off, ln) for off, ln in cl[half:]], C.CALL)
    g.close()
    for a, b in zip(got, rest):
        a["status"] += b["status"]
        a["frames"] += b["frames"]
    _assert_match(got, _oracle(pyref, mode, iq, cfg, cl, C.CALL), f"mode {mode} after refused knobs")
    for bad in (dict(signal_l1_nb_samples=0), dict(signal_l1_nb_decimate=0)):
        with pytest.raises(gpu_ctx.DabGpuError) as e:
            gpu_ctx.DabGpu(mode=mode, max_streams=S, ofdm_overrides=bad)
        assert e.value.code == gpu_ctx.ERR_INVALID
