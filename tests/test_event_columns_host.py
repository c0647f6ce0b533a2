"""The per-event result columns without a GPU: the buffers `TraceAnalyzer` allocates for each option set (on the CPU),
the names, order, dtypes and trailing shapes of `AnalysisResult.columns` (the keys of `tables_to_host` and
`StreamResult.tables`), and the `LevelTable` / `StepFitTable` helpers the analyzer's step relies on."""
import numpy as np
import pytest
import torch

from cusumtools_b200 import cusum, detect, pipeline, synth

CAP, NK, ML, K = 64, 40, 16, 8
EVENT = [("starts", torch.int64, ()), ("ends", torch.int64, ()), ("types", torch.int32, ())]
LEVELS = [("n_levels", torch.int32, ()), ("edges", torch.int32, (ML + 1,)), ("mean", torch.float64, (ML,)),
          ("std", torch.float64, (ML,)), ("overflow", torch.uint8, ())]
INTRA = [("intra_count", torch.int32, ()), ("intra_pairs", torch.int32, (2 * K,))]
FIT = [("stepfit_params", torch.float64, (6,)), ("stepfit_cost", torch.float64, ()), ("stepfit_iters", torch.int32, ())]
CUSUM = {"cusum_delta": 400.0, "cusum_h": 10.0}
OPTION_SETS = {
    "detect": ({}, EVENT),
    "cusum": (CUSUM, EVENT + LEVELS),
    "cusum_intra": ({**CUSUM, "intra_threshold": 40.0, "intra_hysteresis": 4.0}, EVENT + LEVELS + INTRA),
    "stepfit_only": ({"stepfit_samples": 500}, EVENT + LEVELS + FIT),
    "all": ({**CUSUM, "intra_threshold": 40.0, "intra_hysteresis": 4.0, "stepfit_samples": 500, "stepfit_fallback": True},
            EVENT + LEVELS + INTRA + FIT),
}


def _analyzer(opts):
    return pipeline.TraceAnalyzer(1 << 20, synth.CHIMERA_SETTINGS, 1e5, 8, baseline_min=4700.0, baseline_max=5300.0,
                                  max_levels=ML, max_crossings=K, event_capacity=CAP, device="cpu", **opts)


def _result(an, nk):
    """The AnalysisResult the analyzer's step returns for `nk` events, its columns viewing the analyzer's buffers."""
    return pipeline.AnalysisResult(
        filtered=an.y, detect_trace=an.y, lo_halo=0, baseline=None,
        events=detect.EventList(an.starts[:nk], an.ends[:nk], -1), win_start=an.w0[:nk], win_end=an.w1[:nk],
        types=an.typ[:nk], levels=None if an.levels is None else an.levels.rows(nk), pad_value=0.0, median_codes=(0, 0),
        intra=None if an.intra is None else (an.intra[0][:nk], an.intra[1][:nk]),
        stepfit=None if an.fit is None else an.fit.rows(nk))


@pytest.mark.parametrize("name", list(OPTION_SETS))
def test_columns_of_every_option_set(name):
    opts, want = OPTION_SETS[name]
    an = _analyzer(opts)
    cols = _result(an, NK).columns()
    assert [(k, v.dtype, tuple(v.shape)) for k, v in cols.items()] == [(k, dt, (NK,) + s) for k, dt, s in want]
    assert (an.levels is None) == ("n_levels" not in cols) and (an.fit is None) == ("stepfit_params" not in cols)
    assert (an.intra is None) == ("intra_count" not in cols)
    # with an index offset only starts and ends are new tensors
    an.starts.copy_(torch.arange(CAP))
    an.ends.copy_(torch.arange(CAP) + 5)
    moved = _result(an, NK).columns(1000)
    assert list(moved) == list(cols)
    assert torch.equal(moved["starts"], torch.arange(NK) + 1000) and torch.equal(moved["ends"], torch.arange(NK) + 1005)
    for k in list(cols)[2:]:
        assert moved[k].data_ptr() == cols[k].data_ptr(), k


def test_rows_are_views_of_the_capacity_buffers():
    an = _analyzer(OPTION_SETS["all"][0])
    lv, fit = an.levels.rows(NK), an.fit.rows(NK)
    for f in ("n_levels", "edges", "mean", "std", "overflow"):
        part, whole = getattr(lv, f), getattr(an.levels, f)
        assert part.data_ptr() == whole.data_ptr() and part.shape == (NK,) + whole.shape[1:], f
    assert lv.max_levels == an.levels.max_levels == ML
    for f in ("params", "cost", "iters", "status"):
        part, whole = getattr(fit, f), getattr(an.fit, f)
        assert part.data_ptr() == whole.data_ptr() and part.shape == (NK,) + whole.shape[1:], f
    assert an.fit.status.data_ptr() == an.typ.data_ptr() and an.fit.levels is None and fit.levels is None
    # more events than planned: the tables grow with the other event buffers, the fit status is still the type column
    an._alloc_events(2 * CAP)
    assert an.levels.n_levels.shape == (2 * CAP,) and an.levels.edges.shape == (2 * CAP, ML + 1)
    assert an.fit.params.shape == (2 * CAP, 6) and an.fit.status.data_ptr() == an.typ.data_ptr()
    assert an.intra[1].shape == (2 * CAP, 2 * K) and torch.all(an.intra[1] == -1) and torch.all(an.intra[0] == 0)


def test_clear_leaves_rows_without_levels():
    lv = cusum.LevelTable.empty(CAP, ML, "cpu")
    for buf in (lv.n_levels, lv.edges, lv.overflow):
        buf.fill_(7)
    lv.mean.fill_(1.5)
    lv.std.fill_(2.5)
    lv.clear()
    assert torch.all(lv.n_levels == 0) and torch.all(lv.overflow == 0) and torch.all(lv.edges == -1)
    assert torch.all(lv.mean == 1.5) and torch.all(lv.std == 2.5)             # left as they were


def test_level_rows_back_from_host_columns():
    an = _analyzer(OPTION_SETS["cusum"][0])
    g = torch.Generator().manual_seed(0)
    for buf in (an.levels.n_levels, an.levels.edges, an.levels.overflow, an.starts, an.ends, an.typ):
        buf.copy_(torch.randint(0, 100, buf.shape, generator=g))
    for buf in (an.levels.mean, an.levels.std):
        buf.copy_(torch.randn(buf.shape, generator=g, dtype=torch.float64))
    r = _result(an, NK)
    host = {k: v.numpy() for k, v in r.columns().items()}
    back = cusum.LevelTable.from_columns(host, "cpu")
    assert back.max_levels == ML
    for f in ("n_levels", "edges", "mean", "std", "overflow"):
        assert getattr(back, f).dtype == getattr(r.levels, f).dtype and torch.equal(getattr(back, f), getattr(r.levels, f)), f
    assert np.shares_memory(host["mean"], an.levels.mean.numpy())             # the host columns view the buffers
