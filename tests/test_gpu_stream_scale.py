"""The streamed run (pipeline.StreamingAnalyzer) as bench.py times it, against the oracle chain.

bench.py's `e2e` and `from_file` figures time StreamingAnalyzer over the 2,499,999,600-sample trace of config C2, cut into
E2E_SHARDS time sub-shards: 2^20-sample baseline blocks, a halo of one block, 17 sub-shards of which two start past 2^31,
a reserved head of table rows for the first one, pinned host columns of n // 2048 rows to start with.  Here the same run,
set up from bench.py's own constants, is checked against plain references:
  * the median against a plain count of every code, the filtered trace against the one-call filter and against the
    reference's float64 call sequence around every cut and at both ends of the trace;
  * the baseline table, the events and the CUSUM+ levels against the C twin chain run over the streamed trace itself.
    Inside its owned range a sub-shard saw exactly these float32 samples, so whatever is decided there is equal bit for
    bit.  An event window that crosses a cut was decided partly on the neighbour's halo samples, which differ from the
    neighbour's own by the IIR warm-up and rounding: such events may move by one sample, and their level means by at
    most the largest such difference (measured, and stated with the test's properties);
  * two runs of one analyzer, as the timed loop makes them, are bit for bit the same.
A trace whose first piece gives a poor median estimate makes the run redo the first sub-shard, and a trace with six
events per millisecond makes the pinned host columns grow twice in the middle of the run.  Each case checks the free
device memory first, keeps its device memory under 32 GB and records its peak and its runtime."""
import gc
import time

import numpy as np
import pytest
import torch

import bench
from cusumtools_b200 import filters, pipeline, synth
from oracle import c_twin, events_oracle as eo, trace_oracle as to
from test_gpu_analyzer_steps import _bits, defined
from test_gpu_detect_scale import need

pytestmark = pytest.mark.gpu

S = synth.CHIMERA_SETTINGS
BLOCK, PAD, MINP, MAXP = bench.BASELINE_BLOCK, bench.EVENT_PAD, bench.MINPOINTS, bench.MAXPOINTS
# the keywords bench.py builds its StreamingAnalyzer with
KW = dict(threshold=bench.THRESHOLD, hysteresis=bench.HYSTERESIS, baseline_block=BLOCK, baseline_min=bench.BASELINE_MIN,
          baseline_max=bench.BASELINE_MAX, event_padding=PAD, minpoints=MINP, maxpoints=MAXP, cusum_delta=bench.CUSUM_DELTA,
          cusum_h=bench.CUSUM_H)
BASELINE_COLUMNS = ("cnt", "s1", "s2", "mean", "std", "sign", "t_start", "t_end")
CHUNK = 1 << 28


@pytest.fixture(autouse=True)
def peak_and_runtime(record_property):
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    yield
    torch.cuda.synchronize()
    record_property("runtime_s", round(time.perf_counter() - t0, 1))
    record_property("max_memory_allocated_GB", round(torch.cuda.max_memory_allocated() / 1e9, 2))
    gc.collect()
    torch.cuda.empty_cache()


def code_hist(codes: torch.Tensor) -> np.ndarray:
    """Plain count of every masked code (as bench.py's parity check makes it)."""
    mask = filters.chimera_bitmask(S)
    hist = torch.zeros(65536, dtype=torch.int64, device=codes.device)
    for a in range(0, codes.numel(), CHUNK):
        hist += torch.bincount(codes[a:a + CHUNK].to(torch.int32) & mask, minlength=65536)
    return hist.cpu().numpy()


def exact_pair(hist: np.ndarray) -> tuple[int, int]:
    cdf = np.cumsum(hist)
    ntot = int(cdf[-1])
    return int(np.searchsorted(cdf, (ntot - 1) // 2 + 1)), int(np.searchsorted(cdf, ntot // 2 + 1))


def pinned_trace(n: int, **kw):
    """synth.device_trace copied once into pinned host memory, and the count of its codes; nothing left on the device."""
    raw = synth.device_trace(n, torch.device("cuda"), **kw)
    hist = code_hist(raw)
    host = torch.empty(n, dtype=torch.uint16, pin_memory=True)
    host.copy_(raw)
    del raw
    torch.cuda.empty_cache()
    return host, hist


def max_abs_diff(dev: torch.Tensor, host: np.ndarray) -> float:
    """max |dev - host| over two float32 vectors of the same length, on the device, piece by piece."""
    worst = 0.0
    for a in range(0, dev.numel(), CHUNK):
        b = min(dev.numel(), a + CHUNK)
        worst = max(worst, (dev[a:b] - torch.from_numpy(host[a:b]).cuda()).abs().max().item())
    return worst


def run_twice(host: torch.Tensor) -> dict:
    """Two runs of one StreamingAnalyzer over `host`, as bench.py's timed loop makes them.  Everything the checks need
    from the first run is copied out before the second (its tables are views of pinned buffers the next run reuses),
    the second must equal it bit for bit, and the analyzer is released before returning."""
    n = host.numel()
    san = pipeline.StreamingAnalyzer(n, S, bench.CUTOFF, bench.ORDER, shards=bench.E2E_SHARDS, **KW)
    runs = []
    for _ in range(2):
        r = san.run_from_host(host)
        runs.append(dict(tables={k: v.copy() for k, v in r.tables.items()},
                         baseline={k: r.baseline.dev[k].cpu().numpy() for k in BASELINE_COLUMNS},
                         scalars=(tuple(r.median_codes), r.pad_value, r.first_event_id, r.total_events, r.redone)))
        if len(runs) == 1:
            yh = r.filtered.cpu().numpy()
            c0, shift = r.baseline.dev["c0"], r.baseline.dev["shift"]
        else:
            for a in range(0, n, CHUNK):
                b = min(n, a + CHUNK)
                assert torch.equal(r.filtered[a:b].view(torch.int32), torch.from_numpy(yh[a:b]).cuda().view(torch.int32)), a
        del r
    first, second = runs
    assert second["scalars"] == first["scalars"]
    for k in BASELINE_COLUMNS:
        assert np.array_equal(_bits(second["baseline"][k]), _bits(first["baseline"][k])), k
    t1, t2 = defined(first["tables"]), defined(second["tables"])
    assert list(t1) == list(t2)
    for k in t1:
        assert t1[k].dtype == t2[k].dtype and np.array_equal(_bits(t1[k]), _bits(t2[k])), k
    out = dict(first, y=yh, c0=c0, shift=shift, sub=list(san.sub), h=san.h, pin_rows=san._pin["starts"].shape[0],
               halo_diff=halo_differences(san, yh))
    del san
    gc.collect()
    torch.cuda.empty_cache()
    return out


def halo_differences(san, yh: np.ndarray) -> dict:
    """{cut: max |a sub-shard's own sample - the neighbour's owned sample|} over the halo samples within one event
    window (maxpoints + 2 padding) of the cut.  Sub-shards of one shape share an analyzer, which keeps the detection
    trace of the last one it ran: the first sub-shard's right halo, both halos of the last full-length one and the last
    one's left halo, at three cuts (at the benchmark's shape, two of them past 2^31)."""
    reach = MAXP + 2 * PAD
    last = {(eb - ea, a - ea, eb - b): k for k, (a, b, ea, eb) in enumerate(san.sub)}
    out = {}
    for key, k in last.items():
        a, b, ea, eb = san.sub[k]
        y = san.analyzers[key].y
        for lo, hi, cut in ((max(ea, a - reach), a, a), (b, min(eb, b + reach), b)):
            if hi > lo:
                out[cut] = max(out.get(cut, 0.0), max_abs_diff(y[lo - ea:hi - ea], yh[lo:hi]))
    return out


def one_call_differences(host: torch.Tensor, med, yh: np.ndarray, cuts, h: int, lim: int):
    """The streamed trace against filters.dequant_filtfilt over the whole trace with the exact median: the largest
    difference over [0, lim) and within h of each cut below lim."""
    raw = host.cuda()
    ref = filters.dequant_filtfilt(raw, S, bench.CUTOFF, bench.ORDER, median_codes=med)
    del raw
    worst = max_abs_diff(ref[:lim], yh[:lim])
    near = {c: max_abs_diff(ref[c - h:min(lim, c + h)], yh[c - h:min(lim, c + h)]) for c in cuts if c < lim}
    del ref
    torch.cuda.empty_cache()
    return worst, near


def reference_windows(codes: np.ndarray, yh: np.ndarray, pad_value: float, points) -> dict:
    """The reference's call sequence (plot-trace.py:313-320: float64, scipy filtfilt, constant pad = the global
    median's current) over the two blocks around each point, with 8192 samples of margin that keep the window's own
    ends out of reach; at a true end of the trace the window's pad is the trace's.  Largest difference per point."""
    from scipy.signal import bessel, filtfilt
    n = codes.size
    b_, a_ = bessel(bench.ORDER, 2.0 * bench.CUTOFF / np.floor(np.squeeze(S["ADCSAMPLERATE"])), "low")
    out = {}
    for c in points:
        p0, p1 = max(0, c - BLOCK), min(n, c + BLOCK)
        q0, q1 = max(0, p0 - 8192), min(n, p1 + 8192)
        x = to.scale_raw_data(codes[q0:q1], S)
        y_ref = filtfilt(b_, a_, np.pad(x, 1000, mode="constant", constant_values=pad_value), padtype=None)[1000:-1000]
        lo = 0 if q0 == 0 else p0 - q0
        hi = q1 - q0 if q1 == n else p1 - q0
        out[c] = float(np.abs(yh[q0 + lo:q0 + hi].astype(np.float64) - y_ref[lo:hi]).max())
    return out


def check_baseline(run: dict, lim: int):
    """Every block below lim, the partial last one included, against c_twin.block_stats -> baseline_from_stats ->
    thresholds over the streamed trace; returns the oracle's detector lines."""
    yh, bl = run["y"], run["baseline"]
    nb = -(-lim // BLOCK)
    cnt, s1, s2 = c_twin.block_stats(yh[:lim], BLOCK, bench.BASELINE_MIN, bench.BASELINE_MAX, np.float32(run["c0"]),
                                     run["shift"])
    assert np.all(cnt >= 16)                   # no block inherits: a sub-shard's first block has its own row
    mean, std = eo.baseline_from_stats(cnt, s1, s2, run["c0"], run["shift"])
    sign, ts, te = eo.thresholds(mean, std, bench.THRESHOLD, bench.HYSTERESIS)
    for k, want in zip(BASELINE_COLUMNS, (cnt, s1, s2, mean, std, sign, ts, te)):
        assert np.array_equal(bl[k][:nb], want), k
    return sign, ts, te


def owned_inside(w0, w1, sub) -> np.ndarray:
    """Windows [w0, w1) that lie inside one sub-shard's owned range (a window that leaves the trace is clipped to it)."""
    w0, w1 = np.maximum(w0, sub[0][0]), np.minimum(w1, sub[-1][1])
    inside = np.zeros(w0.size, dtype=bool)
    for a, b, _, _ in sub:
        inside |= (w0 >= a) & (w1 <= b)
    return inside


def check_events(run: dict, lines, lim: int, margin: int) -> dict:
    """The streamed event table against c_twin.detect_events + eo.event_windows over the streamed trace: events with a
    window inside one owned range equal, the others (across a cut) each present once with start and end within one
    sample, on the events that start before lim - margin."""
    t, yh, n = run["tables"], run["y"], run["y"].size
    gs, ge, gt = t["starts"], t["ends"], t["types"]
    assert gs.size == run["scalars"][3] and run["scalars"][2] == 0          # total_events, first_event_id
    assert np.all(np.diff(gs) > 0) and gs[0] >= 0 and gs[-1] < n          # so each lies in exactly one owned range
    s, e, _ = c_twin.detect_events(yh[:lim], BLOCK, *lines, cap=4_000_000)
    w0, w1, typ = eo.event_windows(s, e, lim, PAD, MINP, MAXP)
    k, g = s < lim - margin, gs < lim - margin
    s, e, typ, w0, w1, gs, ge, gt = s[k], e[k], typ[k], w0[k], w1[k], gs[g], ge[g], gt[g]
    assert gs.size == s.size
    inside = owned_inside(w0, w1, run["sub"])
    assert np.array_equal(gs[inside], s[inside]) and np.array_equal(ge[inside], e[inside])
    assert np.array_equal(gt[inside], typ[inside])
    ds, de = np.abs(gs - s)[~inside], np.abs(ge - e)[~inside]
    assert ds.max(initial=0) <= 1 and de.max(initial=0) <= 1
    return dict(events=int(s.size), exact=int(inside.sum()), across_cuts=int((~inside).sum()),
                across_moved=int(((ds > 0) | (de > 0)).sum()), past_2p31=int((s >= 1 << 31).sum()))


def check_levels(run: dict, lim: int, margin: int, tol: float) -> dict:
    """CUSUM+ of every accepted event within 2h of a cut and every 97th of the others (events starting below
    lim - margin) against c_twin.cusum_batch over the streamed trace's windows: equal inside one owned range; across
    a cut the same n_levels, edges within one sample and, where the edges agree, means and stds within `tol`."""
    t, yh = run["tables"], run["y"]
    gs, ge, gt = t["starts"], t["ends"], t["types"]
    cuts = np.array([a for a, _, _, _ in run["sub"][1:]], dtype=np.int64)
    idx = np.arange(gs.size)
    near = np.abs(gs[:, None] - cuts[None, :]).min(axis=1) < 2 * run["h"]
    rows = idx[(gt == 0) & (near | (idx % 97 == 0)) & (gs < lim - margin)]
    w0, w1 = gs[rows] - PAD, ge[rows] + PAD
    max_levels = t["mean"].shape[1]
    offs = np.concatenate(([0], np.cumsum(w1 - w0)))
    flat = np.concatenate([yh[a:b] for a, b in zip(w0, w1)])
    nl, ed, mu, sd, ov = c_twin.cusum_batch(flat, offs, bench.CUSUM_DELTA, bench.CUSUM_H, max_levels)
    g = {k: t[k][rows] for k in ("n_levels", "edges", "mean", "std", "overflow")}
    used = np.arange(max_levels)[None, :] < nl[:, None]
    inside = owned_inside(w0, w1, run["sub"])
    assert np.array_equal(g["n_levels"], nl)
    ui = used[inside]
    assert np.array_equal(g["edges"][inside], ed[inside]) and np.array_equal(g["overflow"][inside], ov[inside])
    assert np.array_equal(g["mean"][inside][ui], mu[inside][ui]) and np.array_equal(g["std"][inside][ui], sd[inside][ui])
    x = ~inside
    assert np.abs(g["edges"][x] - ed[x]).max(initial=0) <= 1
    same_edges = x & np.all(g["edges"] == ed, axis=1)
    us = used[same_edges]
    dm = np.abs(g["mean"][same_edges][us] - mu[same_edges][us]).max(initial=0.0)
    dsd = np.abs(g["std"][same_edges][us] - sd[same_edges][us]).max(initial=0.0)
    assert dm <= tol and dsd <= tol, (dm, dsd, tol)
    return dict(rows=int(rows.size), rows_exact=int(inside.sum()), levels_exact=int(nl[inside].sum()),
                rows_across_cuts=int(x.sum()), edges_moved=int((x & ~same_edges).sum()), level_mean_diff_pA=float(dm),
                level_std_diff_pA=float(dsd), tolerance_pA=tol, past_2p31=int((w0 >= 1 << 31).sum()))


def check_run(run: dict, host: torch.Tensor, hist: np.ndarray, lim: int, margin: int, record_property) -> dict:
    """All oracle checks of a streamed run over [0, lim) (the whole trace when lim = n)."""
    n, sub, h = host.numel(), run["sub"], run["h"]
    cuts = [a for a, _, _, _ in sub[1:]]
    med, pad_value = run["scalars"][0], run["scalars"][1]
    assert med == exact_pair(hist)
    assert pad_value == float(np.median(to.scale_raw_data(np.array(med, dtype=np.uint16), S)))
    # the filtered trace: the one-call filter everywhere, the reference's call sequence around the cuts and the ends
    worst, near = one_call_differences(host, med, run["y"], cuts, h, lim)
    assert worst < 0.02, worst
    ref = reference_windows(host.numpy(), run["y"], pad_value, [0] + [c for c in cuts if c < lim] + ([n] if lim == n else []))
    assert max(ref.values()) < 0.05, ref
    lines = check_baseline(run, lim)
    ev = check_events(run, lines, lim, margin)
    # the level means of an event across a cut move by at most the largest difference between the halo samples it
    # used and the neighbour's owned ones; that difference is measured at three cuts, twice it covers the others
    tol = 2.0 * max(run["halo_diff"].values()) + 1e-9
    lv = check_levels(run, lim, margin, tol)
    props = dict(redone=run["scalars"][4], median_codes=list(med), max_diff_one_call_pA=worst,
                 max_diff_within_h_of_cut_pA={int(c): round(v, 6) for c, v in near.items()},
                 max_diff_reference_pA={int(c): round(v, 6) for c, v in ref.items()},
                 halo_diff_pA={int(c): v for c, v in run["halo_diff"].items()}, events=ev, levels=lv)
    for k, v in props.items():
        record_property(k, v)
    return props


def test_streamed_run_at_the_benchmark_step(record_property):
    """bench.py's e2e run: config C2's trace from pinned host memory through StreamingAnalyzer with E2E_SHARDS,
    twice, against the oracle chain over the whole trace."""
    need(32e9)
    n = bench.C2_SAMPLES
    host, hist = pinned_trace(n, seed=1234)
    run = run_twice(host)
    # the layout the benchmark runs: a first sub-shard of four blocks, 15 of 149 blocks, a last one ending in a
    # partial block; two cuts past 2^31
    h, per = 1 << 20, 149 * BLOCK
    assert run["h"] == h
    want = [(0, 4 * BLOCK)] + [(4 * BLOCK + i * per, 4 * BLOCK + (i + 1) * per) for i in range(15)]
    want.append((want[-1][1], n))
    assert [(a, b) for a, b, _, _ in run["sub"]] == want and n - want[-1][0] == 152_237_936
    assert [(ea, eb) for a, b, ea, eb in run["sub"]] == [(max(0, a - h), min(n, b + h)) for a, b in want]
    assert [a for a, _ in want if a > 1 << 31] == [2_191_523_840, 2_347_761_664]
    assert run["pin_rows"] == n // 2048 and run["scalars"][4] in ("", "first")
    props = check_run(run, host, hist, n, 0, record_property)
    assert props["events"]["past_2p31"] > 0 and props["levels"]["past_2p31"] > 0


def test_streamed_run_redoes_the_first_sub_shard(record_property):
    """The codes of the first arrival (the first sub-shard and its right halo) sit 16 code steps higher, so the
    estimate from it misses the median and the first sub-shard is redone with the exact pad: its rows are written
    again, right-aligned in the reserved head.  Median, pad, the filtered trace at the start and at the first cut and
    the tables over the first two sub-shards against the oracle chain."""
    need(32e9)
    n = bench.C2_SAMPLES
    host, hist = pinned_trace(n, seed=1234)
    first_arrival = 4 * BLOCK + (1 << 20)                  # san.sub[0][3], checked below
    head = host.numpy()[:first_arrival]
    mask = filters.chimera_bitmask(S)
    hist -= np.bincount(head & mask, minlength=65536)
    head += np.uint16(64)
    hist += np.bincount(head & mask, minlength=65536)
    run = run_twice(host)
    assert run["sub"][0][3] == first_arrival and run["scalars"][4] == "first"
    check_run(run, host, hist, run["sub"][1][1], 4 * (MAXP + 2 * PAD), record_property)


def test_pinned_tables_grow_in_the_middle_of_a_run(record_property):
    """Short pulses six times a millisecond: about 92 000 events against pinned host columns planned for n // 2048 =
    31 250 rows, so they grow twice while the run is in flight (the first sub-shard still fits its reserved head).
    The oracle checks of the benchmark case, and a second run, which grows nothing, equal to the first."""
    need(8e9)
    n = 64_000_000
    host, hist = pinned_trace(n, seed=77, events_per_s=6000, jitter=100, levels=((-1000.0, 150),))
    run = run_twice(host)
    assert run["pin_rows"] == 4 * (n // 2048) and run["scalars"][4] in ("", "first")
    assert run["scalars"][3] > 2 * (n // 2048)
    props = check_run(run, host, hist, n, 0, record_property)
    assert props["levels"]["rows"] > 80_000
