"""One analyzer across many steps, as callers use it: different traces one after another, the median route and the
event capacity changing between steps, steps queued back to back.

`TraceAnalyzer` keeps its histogram, window counts, plan buffer, device median, pinned read buffer and pad-value cache
from step to step, and regrows its per-event buffers when a step finds more events than they hold.  A buffer left stale
by an earlier step, or state that depends on the route or capacity an earlier step took, gives the same values when a
trace is run twice; here every step runs a different trace.  After each step:
  * the median: `median_codes` are the two middle masked codes of the owned samples, `pad_value` is np.median of their
    float64 currents, `last_median` and `last_median_route` say the same;
  * everything else against a fresh analyzer (default capacity, one step) on the same trace, bit for bit: the filtered
    trace, the baseline table, the windows, the open event, the event ids, and every column `tables_to_host` returns
    (taken while CUSUM+ may still run), where defined: level means and stds up to n_levels, crossing pairs up to
    min(count, max_crossings).
The fresh analyzer's own results are pinned by the oracle tests (test_gpu_pipeline.py); what this adds is "no history,
no regrowth".
"""
import contextlib

import numpy as np
import pytest
import torch

import test_gpu_median_plan as mp
from cusumtools_b200 import pipeline, synth
from oracle import trace_oracle as to
from test_gpu_pipeline import _exact_pair

pytestmark = pytest.mark.gpu
S, N = synth.CHIMERA_SETTINGS, mp.N
KW = dict(mp.KW, baseline_block=65536, maxpoints=4000)
CUSUM = dict(cusum_delta=400.0, cusum_h=10.0)
INTRA = dict(intra_threshold=40.0, intra_hysteresis=4.0)
OPTION_SETS = {"detect": {}, "cusum": CUSUM, "cusum+intra": {**CUSUM, **INTRA}, "stepfit_samples": {"stepfit_samples": 500},
               "stepfit_fallback": {**CUSUM, "stepfit_fallback": True}}
# the median route of each trace: the four of test_gpu_median_plan.traces(), then two more c1 traces.  Half the samples
# of the 1240-event trace lie in events, so its median sits in a sparse tail and the estimate is too uncertain (s.e. 2.3
# code steps) for the device window.
MEDIAN_TRACES = ["narrow", "drift", "two levels", "off by two"]
ROUTE = {"narrow": "device", "drift": "host", "two levels": "host after a device miss", "off by two": "device",
         "300 events": "device", "1240 events": "host"}


class Traces:
    """The traces by name, on the host, on the device and pinned, with their median references and the fresh
    analyzer's step on each, computed once."""

    def __init__(self):
        self.codes = mp.traces()
        self.codes["300 events"] = synth.c1_trace(n=N, n_events=300, seed=21)[0]
        self.codes["1240 events"] = synth.c1_trace(n=N, n_events=1240, seed=23)[0]       # one more still open at the end
        self.codes["no baseline"] = self.codes["narrow"] + np.uint16(4096)             # +2.4 nA: no sample in the window
        self._dev, self._median, self._fresh = {}, {}, {}

    def dev(self, name):
        if name not in self._dev:
            self._dev[name] = torch.from_numpy(self.codes[name]).cuda()
        return self._dev[name]

    def median(self, name, lo=0, hi=0):
        key = (name, lo, hi)
        if key not in self._median:
            own = self.codes[name][lo:N - hi]
            self._median[key] = (_exact_pair(own), float(np.median(to.scale_raw_data(own, S))))
        return self._median[key]

    def fresh(self, name, opts, from_host=False):
        key = (name, tuple(sorted(opts.items())), from_host)
        if key not in self._fresh:
            an = pipeline.TraceAnalyzer(N, S, 1e5, 8, **KW, **opts)
            if from_host:
                r = an.run_from_host(torch.from_numpy(self.codes[name]).pin_memory(), chunks=16)
            else:
                r = an.run(self.dev(name))
            self._fresh[key] = snapshot(an, r)
        return self._fresh[key]


@pytest.fixture(scope="module")
def tr():
    return Traces()


def analyzer(**opts):
    return pipeline.TraceAnalyzer(N, S, 1e5, 8, **KW, **opts)


def snapshot(an, r) -> dict:
    """What step `r` of `an` returned, copied out of the analyzer's buffers before its next step.  The host tables are
    taken first, while CUSUM+ may still run."""
    tables = {k: v.copy() for k, v in an.tables_to_host(r).items()}
    bl = r.baseline
    return dict(tables=tables, trace=r.detect_trace.view(torch.int32).clone(),
                windows=(r.win_start.cpu().numpy(), r.win_end.cpu().numpy()),
                baseline={k: np.array(getattr(bl, k)) for k in ("mean", "std", "count", "sign", "t_start", "t_end")},
                scalars=(r.events.open_start, r.first_event_id, r.total_events, r.median_codes, r.pad_value))


def stream_snapshot(r) -> dict:
    bl = r.baseline
    return dict(tables={k: v.copy() for k, v in r.tables.items()}, trace=r.filtered.view(torch.int32).clone(),
                baseline={k: np.array(getattr(bl, k)) for k in ("mean", "std", "count", "sign", "t_start", "t_end")},
                scalars=(r.first_event_id, r.total_events, tuple(r.median_codes), r.pad_value, r.redone))


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view({8: np.int64, 4: np.int32}[a.itemsize]) if a.dtype.kind == "f" else a


def defined(tables: dict) -> dict:
    """The columns with their undefined entries zeroed: level means and stds past n_levels, crossing pairs past
    min(count, max_crossings)."""
    out = dict(tables)
    if "n_levels" in tables:
        m = np.arange(tables["mean"].shape[1])[None, :] < tables["n_levels"][:, None]
        out["mean"], out["std"] = np.where(m, tables["mean"], 0.0), np.where(m, tables["std"], 0.0)
    if "intra_count" in tables:
        k = tables["intra_pairs"].shape[1]
        m = np.arange(k)[None, :] < 2 * np.minimum(tables["intra_count"], k // 2)[:, None]
        out["intra_pairs"] = np.where(m, tables["intra_pairs"], 0)
    return out


def same(got: dict, want: dict, what) -> None:
    assert got["scalars"] == want["scalars"], what
    assert torch.equal(got["trace"], want["trace"]), what
    for k in want["baseline"]:
        assert np.array_equal(_bits(got["baseline"][k]), _bits(want["baseline"][k])), (what, k)
    for x, y in zip(got.get("windows", ()), want.get("windows", ())):
        assert np.array_equal(x, y), what
    a, b = defined(got["tables"]), defined(want["tables"])
    assert list(a) == list(b), what
    for k in b:
        assert a[k].dtype == b[k].dtype and a[k].shape == b[k].shape, (what, k)
        assert np.array_equal(_bits(a[k]), _bits(b[k])), (what, k)


def check_median(tr, an, r, name, route, lo=0, hi=0) -> None:
    pair, pad = tr.median(name, lo, hi)
    assert r.median_codes == pair and an.last_median == pair, (name, r.median_codes, pair)
    assert r.pad_value == pad, name
    assert an.last_median_route == route, name


@pytest.mark.parametrize("name, fused, halo", [(n, f, 0) for n in MEDIAN_TRACES for f in (True, False)]
                         + [("narrow", True, 131072), ("off by two", False, 131072)])
def test_regrowth_keeps_the_median_on_every_route(tr, name, fused, halo):
    """A first step with more events than the 16 planned regrows the event buffers and redoes detection; the device
    median written before that must be the one the step returns (the two-level trace has no event: no regrowth)."""
    opts = dict(CUSUM, fused_count=fused, lo_halo=halo, hi_halo=halo)
    an = analyzer(event_capacity=16, **opts)
    r = an.run(tr.dev(name))
    check_median(tr, an, r, name, ROUTE[name], halo, halo)
    assert (an.cap > 16) == (name != "two levels"), an.cap
    same(snapshot(an, r), tr.fresh(name, opts), name)


SEQUENCE = ["300 events", "narrow", "drift", "two levels", "off by two", "1240 events", "no baseline", "narrow"]


@pytest.mark.parametrize("option_set", list(OPTION_SETS))
def test_one_analyzer_over_a_sequence_of_traces(tr, option_set):
    """Eight steps through one analyzer planned for 300 events: it grows at the second step and again at the sixth,
    the median route changes from step to step, the seventh trace has no valid baseline block and raises, and the
    analyzer carries on."""
    opts = OPTION_SETS[option_set]
    an = analyzer(event_capacity=300, **opts)
    caps = []
    for i, name in enumerate(SEQUENCE):
        what = (option_set, i, name)
        if name == "no baseline":
            for a in (an, analyzer(**opts)):
                with pytest.raises(ValueError, match="no baseline block"):
                    a.run(tr.dev(name))
            continue
        r = an.run(tr.dev(name))
        check_median(tr, an, r, name, ROUTE[name])
        caps.append(an.cap)
        same(snapshot(an, r), tr.fresh(name, opts), what)
    assert caps[0] == 300 and caps[1] > 300 and caps[4] == caps[1] and caps[5] > caps[4], caps


@pytest.mark.parametrize("a, b", [("narrow", "off by two"), ("drift", "narrow"), ("off by two", "two levels")])
def test_back_to_back_steps(tr, a, b):
    """run(A) then run(B) with nothing read in between: B's histogram, count zeroing and planned forward pass queue
    behind A's CUSUM+.  On the default stream and on a side stream, with the same results."""
    opts = dict(CUSUM, **INTRA)
    side = torch.cuda.Stream()
    got = {}
    for where in ("default", "side"):
        an = analyzer(**opts)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side) if where == "side" else contextlib.nullcontext():
            an.run(tr.dev(a))
            r = an.run(tr.dev(b))
            got[where] = snapshot(an, r)
        torch.cuda.current_stream().wait_stream(side)
        check_median(tr, an, r, b, ROUTE[b])
        same(got[where], tr.fresh(b, opts), (a, b, where))
    same(got["side"], got["default"], (a, b))
    # the host tables of each step taken right after its run, while its CUSUM+ may still run
    an = analyzer(**opts)
    for name in (a, b, a):
        r = an.run(tr.dev(name))
        same(snapshot(an, r), tr.fresh(name, opts), (a, b, name))


def test_run_from_host_sequence(tr):
    """run_from_host (chunked copy, estimate from the first chunk, host-side median) through one analyzer planned for
    16 events, over three traces."""
    an = analyzer(event_capacity=16, **CUSUM)
    for name in ("narrow", "drift", "off by two"):
        r = an.run_from_host(torch.from_numpy(tr.codes[name]).pin_memory(), chunks=16)
        check_median(tr, an, r, name, "host")
        same(snapshot(an, r), tr.fresh(name, CUSUM, from_host=True), name)


def test_streaming_analyzer_sequence(tr):
    """One StreamingAnalyzer over a plain trace, one whose first piece gives a poor estimate (the first sub-shard is
    redone), two where a whole sub-shard, halos included, has no baseline sample (the whole-trace analyzer takes
    over, the second time reused), and the plain trace again; each equals a fresh StreamingAnalyzer."""
    kw = dict(KW, **CUSUM)
    san = pipeline.StreamingAnalyzer(N, S, 1e5, 8, shards=5, **kw)
    plain = tr.codes["narrow"]
    first = plain.copy()
    first[:200_000] += np.uint16(64)
    wholes = []
    for k in (2, 3):
        _, _, ea, eb = san.sub[k]
        c = plain.copy()
        c[ea:eb] += np.uint16(4096)
        wholes.append(c)
    for name, codes, redone in (("plain", plain, None), ("first", first, "first"), ("whole 2", wholes[0], "whole"),
                                ("whole 3", wholes[1], "whole"), ("plain again", plain, None)):
        host = torch.from_numpy(codes).pin_memory()
        got = stream_snapshot(san.run_from_host(host))
        want = stream_snapshot(pipeline.StreamingAnalyzer(N, S, 1e5, 8, shards=5, **kw).run_from_host(host))
        if redone:
            assert got["scalars"][4] == redone, name
        assert got["scalars"][2] == _exact_pair(codes), name
        assert got["scalars"][3] == float(np.median(to.scale_raw_data(codes, S))), name
        same(got, want, name)
