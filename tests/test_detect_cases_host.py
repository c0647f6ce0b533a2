"""The detector cases of tests/detect_cases.py mean what they claim, before any kernel runs on them: the segment
reference equals the vectorised definition, the literal state machine and the C twin (the reference of the GPU tests)
on traces the builder materialises on the CPU, and every witness of every case, up to 2^32 samples, holds."""
import numpy as np
import pytest
import torch

import detect_cases as dc
from oracle import c_twin, events_oracle as eo


def oracles(c, y, sequential: bool):
    forms = [eo.detect_events(y, c.block, c.sign, c.t_start, c.t_end, state_in=c.state_in),
             c_twin.detect_events(y, c.block, c.sign, c.t_start, c.t_end, state_in=c.state_in)]
    if sequential:
        forms.append(eo.detect_events_sequential(y, c.block, c.sign, c.t_start, c.t_end, state_in=c.state_in))
    return forms


def assert_same(want, got, what):
    assert np.array_equal(want[0], got[0]) and np.array_equal(want[1], got[1]) and want[2] == got[2], what


@pytest.mark.parametrize("block", [4096, 8192])
@pytest.mark.parametrize("state_in", [False, True])
@pytest.mark.parametrize("n", [1, 2, 31, 4095, 4096, 4097, 8193, 50_000, 300_000])
def test_segment_reference_is_the_definition(n, block, state_in):
    for seed in range(3):
        c = dc.small_case(n, block, state_in, seed=n + seed)
        y = dc.materialise(c, "cpu", seed=seed, chunk=1 << 14).numpy()
        assert dc.symbols_match(c, torch.from_numpy(y), chunk=1 << 14)
        want = dc.reference(c)
        for i, got in enumerate(oracles(c, y, sequential=n <= 50_000)):
            assert_same(want, got, (c.name, i))


@pytest.mark.parametrize("state_in", [False, True])
def test_layout_patterns_on_a_short_trace(state_in):
    """The layout builder at a size the host can materialise: its patterns on run and block boundaries, a long event
    over a whole scan range and a quiet range, all three forms of the definition agreeing with the segment reference."""
    n = 5 * dc.GROUP_SAMPLES + 77
    pts = {k: v for k, v in dc.boundary_points(n, 8192).items() if k in ("run", "range", "block")}
    for rot in range(4):
        c = dc.layout("short", n, 8192, state_in, pts, rot=rot, seed=rot, long_inside=1, quiet_outside=None)
        assert c.witness and [k for k, v in c.witness.items() if not v] == []
        y = dc.materialise(c, "cpu", seed=rot).numpy()
        want = dc.reference(c)
        for i, got in enumerate(oracles(c, y, sequential=False)):
            assert_same(want, got, (rot, i))
    c = dc.layout("quiet", n, 4096, state_in, pts, quiet_outside=1)
    assert [k for k, v in c.witness.items() if not v] == []
    y = dc.materialise(c, "cpu").numpy()
    for got in oracles(c, y, sequential=False):
        assert_same(dc.reference(c), got, "quiet")


@pytest.mark.parametrize("n", dc.SCAN_SIZES + dc.BIG_SIZES)
def test_witnesses_of_the_scale_cases(n):
    for c in dc.scan_cases(n):
        bad = [k for k, v in c.witness.items() if not v]
        assert c.witness and bad == [], (c.name, bad)
        for key in (("long_event_covers_a_whole_scan_range", "quiet_range_has_no_symbol",
                     "open_event_starts_on_the_last_sample", "some_pattern_on_range", "some_pattern_on_block")
                    + (("some_pattern_on_group",) if c.per > 1 else ())):
            assert key in c.witness, (c.name, key)
        if n > 1 << 31:
            assert "some_pattern_on_2^31" in c.witness
        if n > 1 << 32:
            assert "some_pattern_on_2^32" in c.witness
    kinds = {k.split("_on_")[0] + "_on_" + k.split("_on_")[1].split("@")[0]
             for c in dc.scan_cases(n) for k in c.witness if "@" in k}
    cats = {k.split("_on_")[1].split("@")[0] for k in kinds}
    for cat in cats:                        # over the four variants every boundary kind sees every pattern
        assert {f"{p}_on_{cat}" for p in dc.ORDER} <= kinds, cat


def test_scan_shapes():
    assert [dc.scan_shape(n)[1:] for n in dc.SCAN_SIZES] == [(1024, 1), (1025, 2), (2049, 3)]
    assert dc.scan_shape(dc.C2_SAMPLES)[1:] == (9537, 10)


@pytest.mark.parametrize("ts_eq_te", [False, True])
def test_random_traces_agree_in_all_three_forms(ts_eq_te):
    """Random samples against lines that are not crossed (including ts == te): the vectorised definition, the literal
    state machine and the C twin agree."""
    rng = np.random.default_rng(9 + ts_eq_te)
    for n, block in ((1, 4096), (100, 4096), (5000, 4096), (30_000, 8192)):
        nb = -(-n // block)
        sign, ts, te = dc.lines(nb, int(rng.integers(1 << 30)), hysteresis=(0.0,) if ts_eq_te else (0.0, 1.0, 3.0))
        lo = np.minimum(sign * ts, sign * te).astype(np.float64) - 20
        hi = np.maximum(sign * ts, sign * te).astype(np.float64) + 20
        kb = np.arange(n) // block
        v = rng.uniform(lo[kb], hi[kb])
        pick = rng.random(n)                      # some samples exactly on a line
        v = np.where(pick < 0.1, (sign * ts)[kb], np.where(pick < 0.2, (sign * te)[kb], v))
        y = (sign[kb] * v).astype(np.float32)
        for state_in in (False, True):
            forms = [eo.detect_events(y, block, sign, ts, te, state_in),
                     eo.detect_events_sequential(y, block, sign, ts, te, state_in),
                     c_twin.detect_events(y, block, sign, ts, te, state_in)]
            for f in forms[1:]:
                assert_same(forms[0], f, (n, state_in))


# ---------------------------------------------------------------------------------- crossed lines are rejected
def test_host_table_rejects_negative_hysteresis():
    from cusumtools_b200 import detect
    bl = detect.Baseline(4096, np.array([100.0, -100.0]), np.ones(2), np.ones(2, np.int64))
    for hys in (-1.0, -1e-12, float("nan")):
        with pytest.raises(ValueError, match="hysteresis"):
            bl.with_thresholds(5.0, hys)
        assert bl._t_start is None and bl._t_end is None
    bl.with_thresholds(5.0, 0.0)
    assert np.array_equal(bl.t_start, bl.t_end)


@pytest.mark.parametrize("kw", [{"hysteresis": -1.0}, {"intra_threshold": 40.0, "intra_hysteresis": -0.5}])
def test_analyzers_reject_negative_hysteresis_before_allocating(kw):
    """Both analyzers refuse crossed lines at construction, before they touch a device (this test runs without one)."""
    from cusumtools_b200 import pipeline, synth
    args = dict(baseline_min=4700.0, baseline_max=5300.0, device="cpu", **kw)
    with pytest.raises(ValueError, match="hysteresis"):
        pipeline.TraceAnalyzer(1 << 20, synth.CHIMERA_SETTINGS, 1e5, 8, **args)
    with pytest.raises(ValueError, match="hysteresis"):
        pipeline.StreamingAnalyzer(1 << 20, synth.CHIMERA_SETTINGS, 1e5, 8, **args)
