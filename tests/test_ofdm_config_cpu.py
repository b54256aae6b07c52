"""Every case of tests/test_ofdm_config_gpu.py has teeth, on the CPU: each synchronisation knob set, live change, Process()
partition and adapter field edit changes what the C restatement computes on at least one recording of its batch, by more than
the GPU comparison tolerates.  A GPU build that ignored the knob or the partition would therefore fail the GPU test.  Where the
reference build exists, the restatement is also compared with it in every case."""
import itertools

import numpy as np
import pytest

import ofdm_config_cases as C


@pytest.fixture(scope="module", params=[1, 2, 3, 4], ids=lambda m: f"mode{m}")
def batch(request):
    mode = request.param
    return mode, C.recordings(mode)


def _frames_desync(run):
    return [(len(r["frames"]), r["status"][-1]["frames_desync"]) for r in run]


def test_knob_sets_change_the_oracle(pyref, batch):
    mode, iq = batch
    cl = C.calls(iq.shape[1] // 2)
    defaults = C.oracle_outputs(pyref, mode, iq, {}, cl, 0)
    base = C.oracle_outputs(pyref, mode, iq, C.BASE[mode], cl, 0)
    assert not C.BASE[mode] or C.differs(defaults, base), "the mode's base knobs change nothing"
    flat = []
    for name in C.knob_cases(mode):
        cfg = C.case_config(name, mode)
        run = C.oracle_outputs(pyref, mode, iq, cfg, cl, 0)
        # ignoring every knob gives the defaults' output, ignoring the case's own knob the base's
        if C.differs(defaults, run) and (cfg == C.BASE[mode] or C.differs(base, run)):
            continue
        flat.append((name, _frames_desync(run)))
    assert not flat, f"mode {mode}: knob sets without effect on the recordings: {flat}"
    assert set(C.KNOBS_C32) <= set(C.KNOBS)


def test_live_changes_change_the_oracle(pyref, batch):
    mode, iq = batch
    cl = C.live_calls(iq.shape[1] // 2)
    base = C.oracle_outputs(pyref, mode, iq, C.LIVE_BASE[mode], cl, 0)
    scenarios = C.live_scenarios(mode, base)
    assert set(scenarios) == {"null_search", "mid_frame", "after_desync", "coarse_toggle"}
    for name, edits in scenarios.items():
        assert all(0 < k < len(cl) for k in edits)
        run = C.oracle_outputs(pyref, mode, iq, C.LIVE_BASE[mode], cl, 0, edits=edits)
        assert C.differs(base, run), f"mode {mode}: live change {name} at calls {sorted(edits)} changes nothing"


def test_partitions_change_the_oracle(pyref, batch):
    """Each partition against blocks of CALL samples over the same stretch, at the base knobs and at PARTITION_KNOBS"""
    mode, iq = batch
    n = iq.shape[1] // 2
    flat = []
    for c32 in (False, True):
        for pname, k in C.partition_cases(mode, c32):
            lengths, bs, limit = C.partitions(mode)[pname]
            cfg = C.BASE[mode] if k is None else C.case_config(k, mode)
            ref = C.oracle_outputs(pyref, mode, iq, cfg, C.partition_calls(n, [C.CALL], limit), 0)
            run = C.oracle_outputs(pyref, mode, iq, cfg, C.partition_calls(n, lengths, limit), bs)
            if not C.differs(ref, run, per_call=False):
                flat.append((pname, k))
    assert not flat, f"mode {mode}: partitions without effect: {flat}"


def test_partition_rings_hold_their_blocks(dab):
    for mode in (1, 2, 3, 4):
        P = dab.get_params(mode)
        for pname, (lengths, bs, _) in C.partitions(mode).items():
            ring = C.ring_for_block(mode, bs or max(lengths))
            assert ring & (ring - 1) == 0
            assert ring - P.nb_frame_samples - P.nb_null_period - P.nb_symbol_period - 1024 >= (bs or max(lengths)), (mode, pname)


def test_adapter_field_swaps_change_the_oracle(pyref):
    """Exchanging any two fields of the same type in the adapter's copy of OFDM_Demod_Config changes the output of the edit
    sequence the adapter test runs.  A swap that yields a window of 0 is rejected by the library: the previous knobs stay."""
    mode = C.ADAPTER_MODE
    iq = C.recordings(mode)[list(C.ADAPTER_STREAMS)]
    cl = C.partition_calls(iq.shape[1] // 2, C.ADAPTER_BLOCKS)
    assert max(C.ADAPTER_EDITS) < len(cl)
    base = C.oracle_outputs(pyref, mode, iq, {}, cl, 0, edits=C.ADAPTER_EDITS)
    assert C.differs(C.oracle_outputs(pyref, mode, iq, {}, cl, 0), base)
    for e in C.ADAPTER_EDITS.values():
        assert set(e) == set(C.FLOAT_KNOBS) | set(C.INT_KNOBS) == set(pyref.OFDM_DEFAULTS)
        assert len({e[k] for k in C.FLOAT_KNOBS}) == len(C.FLOAT_KNOBS)
    flat = []
    for group in (C.FLOAT_KNOBS, C.INT_KNOBS):
        for a, b in itertools.combinations(group, 2):
            edits = {k: {**v, a: v[b], b: v[a]} for k, v in C.ADAPTER_EDITS.items()}
            edits = {k: v for k, v in edits.items() if v["signal_l1_nb_samples"] >= 1 and v["signal_l1_nb_decimate"] >= 1}
            if not C.differs(base, C.oracle_outputs(pyref, mode, iq, {}, cl, 0, edits=edits)):
                flat.append((a, b))
    assert not flat, f"field swaps the adapter test would not see: {flat}"


def test_zero_l1_window_is_refused_at_context_creation(dab):
    """dabgpu_ctx_create validates the knobs as dabgpu_ofdm_set_config does, before it looks for a device: a zero-filled
    signal_l1 window (the control kernel divides by both) never reaches a kernel."""
    for bad in (dict(signal_l1_nb_samples=0), dict(signal_l1_nb_decimate=0), dict(signal_l1_nb_samples=-1),
                dict(signal_l1_nb_decimate=-1)):
        with pytest.raises(dab.DabGpuError) as e:
            dab.DabGpu(mode=1, ofdm_overrides=bad)
        assert e.value.code == dab.ERR_INVALID and "signal_l1" in str(e.value)


def test_restatement_matches_reference_under_every_knob_set(pyref, ref_ok, batch):
    """The bar of test_oracle_cpu.py::test_port_vs_reference_ofdm_modes, for every knob set, live change and partition."""
    mode, iq = batch
    n = iq.shape[1] // 2
    runs = [(C.case_config(k, mode), C.calls(n), 0, None) for k in C.knob_cases(mode)]
    live = C.live_calls(n)
    base = C.oracle_outputs(pyref, mode, iq, C.LIVE_BASE[mode], live, 0)
    runs += [(C.LIVE_BASE[mode], live, 0, e) for e in C.live_scenarios(mode, base).values()]
    for pname, k in C.partition_cases(mode):
        lengths, bs, limit = C.partitions(mode)[pname]
        runs.append((C.BASE[mode] if k is None else C.case_config(k, mode), C.partition_calls(n, lengths, limit), bs, None))
    for cfg, cl, bs, edits in runs:
        port = C.oracle_outputs(pyref, mode, iq, cfg, cl, bs, edits=edits)
        ref = C.oracle_outputs(pyref, mode, iq, cfg, cl, bs, use_ref=True, edits=edits)
        for p, r in zip(port, ref):
            sp, sr = p["status"][-1], r["status"][-1]
            assert (sp["state"], sp["frames_read"], sp["frames_desync"]) == (sr["state"], sr["frames_read"], sr["frames_desync"]), (cfg, bs)
            assert len(p["frames"]) == len(r["frames"]), (cfg, bs)
            for (pb, _, _, pt), (rb, _, _, rt) in zip(p["frames"], r["frames"]):
                assert pt == rt
                assert np.abs(pb.astype(np.int32) - rb.astype(np.int32)).max() <= 1
