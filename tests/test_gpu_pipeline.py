"""GPU parity of the fused single-synchronisation path (pipeline.TraceAnalyzer): baseline
table, detector lines, events, event windows / type codes and CUSUM+ levels against the
oracle chain run on the SAME filtered samples.  Every integer and every float64 table entry
is bit-exact."""
import numpy as np
import pytest
import torch

from cusumtools_b200 import pipeline, synth
from oracle import c_twin, events_oracle as eo

pytestmark = pytest.mark.gpu
S = synth.CHIMERA_SETTINGS
KW = dict(threshold=5.0, hysteresis=1.0, baseline_min=4700.0, baseline_max=5300.0)


def oracle_chain(y, n_keep, block, pad=100, minp=8, maxp=100000, delta=400.0, h=10.0, max_levels=16, lo=0):
    """The oracle's stages 2-3 over the whole detection trace `y`; events whose start lies in
    [lo, lo + n_keep) are kept and reported relative to `lo` (windows stay in `y` coordinates)."""
    c0 = np.float32(5000.0)
    sh = eo.stats_shift(300.0, block)
    cnt, s1, s2 = c_twin.block_stats(y, block, 4700.0, 5300.0, c0, sh)
    mean, std = eo.baseline_from_stats(cnt, s1, s2, c0, sh)
    sign, ts, te = eo.thresholds(mean, std, 5.0, 1.0)
    s, e, o = c_twin.detect_events(y, block, sign, ts, te)
    w0, w1, typ = eo.event_windows(s, e, len(y), pad, minp, maxp)
    keep = (s >= lo) & (s < lo + n_keep)
    s, e, w0, w1, typ = s[keep] - lo, e[keep] - lo, w0[keep], w1[keep], typ[keep]
    o = o - lo if 0 <= o - lo < n_keep else -1
    ok = typ == 0
    offs = np.concatenate(([0], np.cumsum((w1 - w0)[ok])))
    flat = np.concatenate([y[a:b] for a, b in zip(w0[ok], w1[ok])]) if ok.any() else np.zeros(0, np.float32)
    lv = c_twin.cusum_batch(flat, offs, delta, h, max_levels)
    return dict(mean=mean, std=std, sign=sign, ts=ts, te=te, s=s, e=e, o=o, w0=w0, w1=w1, typ=typ, ok=ok, lv=lv)


def check(r, ref):
    assert np.array_equal(r.baseline.mean, ref["mean"]) and np.array_equal(r.baseline.std, ref["std"])
    assert np.array_equal(r.baseline.sign, ref["sign"])
    assert np.array_equal(r.baseline.t_start, ref["ts"]) and np.array_equal(r.baseline.t_end, ref["te"])
    assert np.array_equal(r.events.starts.cpu().numpy(), ref["s"])
    assert np.array_equal(r.events.ends.cpu().numpy(), ref["e"])
    assert np.array_equal(r.win_start.cpu().numpy(), ref["w0"]) and np.array_equal(r.win_end.cpu().numpy(), ref["w1"])
    assert np.array_equal(r.types.cpu().numpy(), ref["typ"])
    ok = ref["ok"]
    nl, ed, mu, sd, ov = ref["lv"]
    gnl = r.levels.n_levels.cpu().numpy()
    assert np.array_equal(gnl[ok], nl) and np.all(gnl[~ok] == 0)
    assert np.array_equal(r.levels.edges.cpu().numpy()[ok], ed)
    L = r.levels.max_levels
    gm, gs = r.levels.mean.cpu().numpy()[ok], r.levels.std.cpu().numpy()[ok]
    for i in range(len(nl)):          # rows are only defined up to n_levels
        assert np.array_equal(gm[i, :nl[i]], mu[i, :nl[i]]) and np.array_equal(gs[i, :nl[i]], sd[i, :nl[i]])
    assert np.array_equal(r.levels.overflow.cpu().numpy()[ok], ov)


@pytest.mark.parametrize("block,cap", [(65536, None), (4096, 5)])
def test_analyzer_matches_oracle_chain(block, cap):
    codes, true_starts = synth.c1_trace(n=600_000, n_events=140, seed=11)
    raw = torch.from_numpy(codes).cuda()
    an = pipeline.TraceAnalyzer(len(codes), S, 1e5, 8, baseline_block=block, cusum_delta=400.0, cusum_h=10.0,
                                event_capacity=cap, **KW)
    for _ in range(2):                       # the second run reuses every buffer
        r = an.run(raw)
        y = r.detect_trace.cpu().numpy()
        ref = oracle_chain(y, len(codes), block)
        check(r, ref)
        assert len(true_starts) <= len(ref["s"]) <= len(true_starts) + 2
        assert r.events.open_start == ref["o"]


def test_analyzer_with_halos_keeps_only_owned_events():
    codes, _ = synth.c1_trace(n=500_000, n_events=115, seed=12)
    lo, hi = 8192, 12288
    raw = torch.from_numpy(codes).cuda()
    an = pipeline.TraceAnalyzer(len(codes), S, 1e5, 8, lo_halo=lo, hi_halo=hi, baseline_block=4096, maxpoints=4000,
                                cusum_delta=400.0, cusum_h=10.0, **KW)
    r = an.run(raw)
    y = r.detect_trace.cpu().numpy()
    assert y.size == len(codes) and r.filtered.numel() == len(codes) - lo - hi and r.lo_halo == lo
    check(r, oracle_chain(y, len(codes) - lo - hi, 4096, lo=lo, maxp=4000))


def test_short_halos_are_rejected():
    """A halo must cover the warm-up of both filter passes and one maximal event window (ADVICE r1): events of
    4k-100k samples straddling a shard boundary would otherwise be dropped or mistyped."""
    with pytest.raises(ValueError, match="shorter than"):
        pipeline.TraceAnalyzer(500_000, S, 1e5, 8, lo_halo=8192, hi_halo=0, baseline_block=4096, **KW)
    with pytest.raises(ValueError, match="shorter than"):
        pipeline.TraceAnalyzer(500_000, S, 1e5, 8, lo_halo=0, hi_halo=65536, baseline_block=4096, **KW)
    pipeline.TraceAnalyzer(500_000, S, 1e5, 8, lo_halo=0, hi_halo=65536, baseline_block=4096, maxpoints=50_000, **KW)


def test_no_valid_baseline_block_raises():
    codes, _ = synth.c1_trace(n=100_000, n_events=10, seed=3)
    an = pipeline.TraceAnalyzer(len(codes), S, 1e5, 8, baseline_block=4096, threshold=5.0, hysteresis=1.0,
                                baseline_min=100.0, baseline_max=200.0)
    with pytest.raises(ValueError):
        an.run(torch.from_numpy(codes).cuda())


def test_event_table_and_analysis_dir_from_the_gpu_path(tmp_path):
    import pandas as pd
    from cusumtools_b200 import writer
    codes, true_starts = synth.c1_trace(n=400_000, n_events=95, seed=13)
    an = pipeline.TraceAnalyzer(len(codes), S, 1e5, 8, baseline_block=65536, cusum_delta=400.0, cusum_h=10.0, **KW)
    r = an.run(torch.from_numpy(codes).cuda())
    y = r.detect_trace.cpu().numpy()
    lo, hi = writer.event_extrema(r.detect_trace, r.win_start, r.win_end)
    w0, w1 = r.win_start.cpu().numpy(), r.win_end.cpu().numpy()
    assert np.array_equal(lo.cpu().numpy(), [y[max(a, 0):b].min() for a, b in zip(w0, w1)])
    assert np.array_equal(hi.cpu().numpy(), [y[max(a, 0):b].max() for a, b in zip(w0, w1)])
    tab = writer.event_table_from_result(an, r, samplerate=synth.FS)
    assert len(true_starts) - 1 <= len(tab) <= len(true_starts)
    # the 100-sample baseline paddings contain part of the filtered edges, so blockages read a little low
    assert abs(np.median(tab.events["max_blockage_pA"]) - 1600) < 100 and np.median(tab.events["n_levels"]) in (3, 4)
    assert np.all(np.abs(tab.events["start_time_s"] - (true_starts[:len(tab)] + 0.0) / synth.FS) < 60 / synth.FS)
    ids = tab.events["id"][:3]
    out = str(tmp_path / "an")
    writer.write_analysis_dir(out, tab, baseline_mean=r.baseline.mean, baseline_std=r.baseline.std, baseline_block=an.block,
                              samplerate=synth.FS, threshold=5.0, hysteresis=1.0, cutoff=1e5, poles=8,
                              event_samples=writer.gather_event_samples(an, r, ids, tab))
    db = pd.read_csv(out + "/events.csv")
    assert len(db) == len(tab) and list(db.columns) == writer.EVENT_COLUMNS
    ef = pd.read_csv(out + "/events/event_%08d.csv" % ids[0])
    i = int(ids[0])
    assert np.allclose(ef["current_pA"].values, y[w0[i]:w1[i]])
    assert set(np.round(ef["cusum_fit"].values, 6)) == set(np.round(r.levels.mean.cpu().numpy()[i, :r.levels.n_levels[i].item()], 6))


@pytest.mark.parametrize("origin", [0, 8192, 70000])
def test_block_sums_fused_into_the_filter_equal_the_standalone_kernel(origin):
    """The filter's epilogue tallies the same exact integer sums as ct_block_stats_f32, for any
    origin of the block grid (time shards start it after their left halo)."""
    from cusumtools_b200 import detect, filters
    from cusumtools_b200.design import bessel_lowpass
    codes, _ = synth.c1_trace(n=900_000, n_events=200, seed=17)
    raw = torch.from_numpy(codes).cuda()
    g = filters.stats_granule(len(codes), 1000, bessel_lowpass(8, 2 * 1e5 / synth.FS))
    block = g * max(2, 65536 // g)             # a whole number of warp groups, at least 65536 samples
    n_det = len(codes) - origin
    bl = detect.new_baseline(n_det, block, 4700.0, 5300.0, raw.device)
    y = filters.dequant_filtfilt(raw, S, 1e5, 8, stats=detect.stats_args(bl, origin=origin))
    y0 = filters.dequant_filtfilt(raw, S, 1e5, 8)
    assert torch.max(torch.abs(y - y0)).item() < 0.01     # the shifted run grid changes the samples only by rounding
    ref = detect.baseline_blocks(y[origin:], block, 4700.0, 5300.0)
    for k in ("cnt", "s1", "s2"):
        assert torch.equal(bl.dev[k], ref.dev[k]), k


def test_fused_block_sums_refuse_small_blocks():
    from cusumtools_b200 import detect, filters
    from cusumtools_b200.design import bessel_lowpass
    codes, _ = synth.c1_trace(n=900_000, n_events=200, seed=17)
    raw = torch.from_numpy(codes).cuda()
    g = filters.stats_granule(len(codes), 1000, bessel_lowpass(8, 2 * 1e5 / synth.FS))
    if g >= 65536:
        pytest.skip("the run grid of this trace is already coarser than the limit")
    bl = detect.new_baseline(len(codes), g, 4700.0, 5300.0, raw.device)
    with pytest.raises(RuntimeError, match="at least 65536"):
        filters.dequant_filtfilt(raw, S, 1e5, 8, stats=detect.stats_args(bl, origin=0))


@pytest.mark.parametrize("n,lo,hi", [(300_001, 0, 0), (300_000, 0, 0), (5_000_000, 0, 0), (5_000_001, 65536, 8192)])
def test_analyzer_filter_with_estimated_median_matches_the_oracle_at_the_trace_ends(n, lo, hi):
    """The analyzer filters with an ESTIMATED median as subtraction constant, counts the exact
    median on the side and repairs the pad at both ends (pipeline.TraceAnalyzer.run): the result
    must equal the reference's filter_data over the whole trace, ends included, and the median /
    pad value must be the exact ones."""
    from cusumtools_b200 import filters
    from oracle import trace_oracle as to
    codes, _ = synth.c1_trace(n=n, n_events=min(1000, (n - 4000) // synth.EVENT_PERIOD), seed=n % 97)
    raw = torch.from_numpy(codes).cuda()
    an = pipeline.TraceAnalyzer(n, S, 1e5, 8, lo_halo=lo, hi_halo=hi, baseline_block=65536, maxpoints=4000,
                                fused_count=(n % 2 == 0), **KW)
    r = an.run(raw)
    own = codes[lo:n - hi]
    srt = np.sort(own & np.uint16(filters.chimera_bitmask(S)))
    assert r.median_codes == (int(srt[(own.size - 1) // 2]), int(srt[own.size // 2]))
    x = to.scale_raw_data(codes, S)
    # the shard's pad value is the median of its OWNED samples (all ranks together: of the whole trace)
    assert r.pad_value == float(np.median(to.scale_raw_data(own, S)))
    want = filters.dequant_filtfilt(raw, S, 1e5, 8, median_codes=r.median_codes).cpu().numpy()   # one-call path, exact median
    got = r.detect_trace.cpu().numpy()
    assert np.abs(got - want).max() < 0.02
    if lo == 0 and hi == 0:
        ref = to.filter_data(x, synth.FS, 1e5, 8)
        assert np.abs(got[:3000] - ref[:3000]).max() < 0.05 and np.abs(got[-3000:] - ref[-3000:]).max() < 0.05
        assert np.abs(got - ref).max() < 0.05


def test_streamed_run_from_host_equals_the_resident_run():
    """run_from_host (chunked copy overlapped with the forward pass, median estimated from the
    first chunk) gives the same events / levels and, to rounding, the same samples as run()."""
    codes, _ = synth.c1_trace(n=3_400_000, n_events=800, seed=31)
    codes[:400_000] += np.uint16(64)          # the first chunk sits 16 codes higher: its median is a poor estimate
    host = torch.from_numpy(codes).pin_memory()
    kw = dict(baseline_block=65536, cusum_delta=400.0, cusum_h=10.0, **KW)
    a = pipeline.TraceAnalyzer(len(codes), S, 1e5, 8, **kw)
    b = pipeline.TraceAnalyzer(len(codes), S, 1e5, 8, **kw)
    ra = a.run(host.cuda())
    for chunks in (3, 16):
        rb = b.run_from_host(host, chunks=chunks)
        assert rb.median_codes == ra.median_codes and rb.pad_value == ra.pad_value
        assert torch.max(torch.abs(ra.filtered - rb.filtered)).item() < 0.02
        assert len(rb.events) == len(ra.events)
        # near-ties may move by one sample
        assert (ra.events.starts - rb.events.starts).abs().max().item() <= 1


@pytest.mark.parametrize("shift_first", [0, 64])
def test_streaming_analyzer_equals_the_resident_run(shift_first):
    """StreamingAnalyzer (time sub-shards processed while the copy is still running, tables sent back per
    sub-shard) against one TraceAnalyzer.run over the whole trace: same medians, same events and levels,
    samples equal to the IIR warm-up error.  With `shift_first` the first piece's median is a poor estimate of
    the global one, so the first sub-shard has to be redone with the exact pad."""
    codes, _ = synth.c1_trace(n=3_400_000, n_events=800, seed=32)
    if shift_first:
        codes[:200_000] += np.uint16(shift_first)
    host = torch.from_numpy(codes).pin_memory()
    kw = dict(baseline_block=65536, cusum_delta=400.0, cusum_h=10.0, **KW)
    a = pipeline.TraceAnalyzer(len(codes), S, 1e5, 8, **kw)
    ra = a.run(host.cuda())
    ta = a.tables_to_host(ra)
    for shards, first_blocks in ((5, 2), (1, 4), (16, 1)):
        b = pipeline.StreamingAnalyzer(len(codes), S, 1e5, 8, shards=shards, first_blocks=first_blocks, **kw)
        for _ in range(2):                                   # buffers are reused from run to run
            rb = b.run_from_host(host)
        assert tuple(rb.median_codes) == tuple(ra.median_codes) and rb.pad_value == ra.pad_value
        if shift_first and shards > 1:
            assert rb.redone == "first"
        assert torch.max(torch.abs(ra.filtered - rb.filtered)).item() < 0.02
        tb = rb.tables
        assert len(tb["starts"]) == len(ta["starts"]) == rb.total_events
        assert np.abs(tb["starts"] - ta["starts"]).max() <= 1 and np.abs(tb["ends"] - ta["ends"]).max() <= 1
        same = (tb["starts"] == ta["starts"]) & (tb["ends"] == ta["ends"])
        assert same.mean() > 0.99
        assert np.array_equal(tb["types"][same], ta["types"][same])
        assert np.array_equal(tb["n_levels"][same], ta["n_levels"][same])
        assert np.mean(np.all(tb["edges"][same] == ta["edges"][same], axis=1)) > 0.99
        bl_a, bl_b = ra.baseline, rb.baseline
        assert len(bl_b) == len(bl_a)
        # a different subtraction constant moves the samples by the float32 DC-gain error (1e-5 of the difference)
        assert np.allclose(bl_b.mean, bl_a.mean, rtol=0, atol=1e-2) and np.allclose(bl_b.std, bl_a.std, rtol=5e-3)
        assert np.array_equal(bl_b.count, bl_a.count) or np.abs(bl_b.count - bl_a.count).max() <= 2


@pytest.mark.parametrize("n", [30_000, 100_000, 700_001])
def test_streaming_analyzer_small_and_ragged_traces(n):
    """Traces shorter than a baseline block, shorter than the first sub-shard, and not a multiple of the block."""
    codes, _ = synth.c1_trace(n=n, n_events=max(2, n // 5000), seed=n)
    host = torch.from_numpy(codes).pin_memory()
    kw = dict(baseline_block=65536, cusum_delta=400.0, cusum_h=10.0, **KW)
    ra_an = pipeline.TraceAnalyzer(n, S, 1e5, 8, **kw)
    ra = ra_an.run(host.cuda())
    ta = ra_an.tables_to_host(ra)
    rb = pipeline.StreamingAnalyzer(n, S, 1e5, 8, shards=16, **kw).run_from_host(host)
    assert tuple(rb.median_codes) == tuple(ra.median_codes)
    assert rb.filtered.numel() == n and torch.max(torch.abs(ra.filtered - rb.filtered)).item() < 0.02
    assert len(rb.tables["starts"]) == len(ta["starts"])
    assert np.abs(rb.tables["starts"] - ta["starts"]).max(initial=0) <= 1
    assert len(rb.baseline) == len(ra.baseline) == -(-n // 65536)


def _tables_agree(ta, tb):
    assert set(ta) == set(tb)
    for k in ("starts", "ends", "types", "n_levels", "overflow", "intra_count"):
        if k in ta:
            assert ta[k].shape == tb[k].shape and np.mean(ta[k] == tb[k]) > 0.98, k
    if "mean" in ta:
        sel = (np.arange(ta["mean"].shape[1])[None, :] < ta["n_levels"][:, None]) & (ta["n_levels"] == tb["n_levels"])[:, None]
        assert not sel.any() or np.mean(ta["edges"][:, 1:][sel] == tb["edges"][:, 1:][sel]) > 0.98
        # The two forms subtract different constants, so their filtered samples differ at the 1e-3 pA level and a
        # decision that sits on a line (an event boundary, a changepoint, a chunk of the in-window rule) can fall either
        # way; level means are compared where the segmentation is the same, which must be (almost) everywhere.
        same = ((ta["starts"] == tb["starts"]) & (ta["ends"] == tb["ends"]) & (ta["n_levels"] == tb["n_levels"])
                & np.all(ta["edges"] == tb["edges"], axis=1))
        assert np.mean(same) > 0.95
        sel &= same[:, None]
        assert np.allclose(ta["mean"][sel], tb["mean"][sel], rtol=0, atol=0.5)


@pytest.mark.parametrize("opts", [
    {}, {"cusum_delta": 400.0, "cusum_h": 10.0}, {"cusum_delta": 400.0, "cusum_h": 10.0, "intra_threshold": 40.0, "intra_hysteresis": 4.0},
    {"intra_threshold": 40.0, "intra_hysteresis": 4.0}, {"cusum_delta": 400.0, "cusum_h": 10.0, "event_capacity": 16},
    {"cusum_delta": 400.0, "cusum_h": 10.0, "max_levels": 3}, {"cusum_delta": 400.0, "cusum_h": 10.0, "maxpoints": 1500}],
    ids=["detect-only", "cusum", "cusum+intra", "intra-only", "regrow", "level-overflow", "too-long"])
def test_streamed_and_resident_forms_agree_for_every_option_set(opts):
    codes, _ = synth.c1_trace(n=2_000_000, n_events=400, seed=9)
    host = torch.from_numpy(codes).pin_memory()
    kw = dict(baseline_block=65536, **KW, **opts)
    a = pipeline.TraceAnalyzer(len(codes), S, 1e5, 8, **kw)
    ta = a.tables_to_host(a.run(host.cuda()))
    rb = pipeline.StreamingAnalyzer(len(codes), S, 1e5, 8, shards=5, **kw).run_from_host(host)
    assert len(ta["starts"]) == 400 and rb.redone in ("", "first")
    _tables_agree(ta, rb.tables)


def test_streaming_analyzer_over_a_shard_with_halos():
    """A rank's extended range [left halo | owned | right halo] through the streamed form: the rows and the
    filtered samples are those of the owned range only, as with TraceAnalyzer."""
    codes, _ = synth.c1_trace(n=2_000_000, n_events=400, seed=9)
    host = torch.from_numpy(codes).pin_memory()
    kw = dict(baseline_block=65536, cusum_delta=400.0, cusum_h=10.0, lo_halo=131072, hi_halo=131072, **KW)
    a = pipeline.TraceAnalyzer(len(codes), S, 1e5, 8, **kw)
    ra = a.run(host.cuda())
    ta = a.tables_to_host(ra)
    rb = pipeline.StreamingAnalyzer(len(codes), S, 1e5, 8, shards=4, **kw).run_from_host(host)
    assert rb.filtered.numel() == len(codes) - 2 * 131072 and rb.redone == ""
    assert torch.max(torch.abs(rb.filtered - ra.filtered)).item() < 0.02
    assert np.array_equal(ta["starts"], rb.tables["starts"]) and np.array_equal(ta["ends"], rb.tables["ends"])


def test_event_table_from_the_streamed_result_equals_the_resident_one():
    """writer.event_table_from_stream over a StreamingAnalyzer result against writer.event_table_from_result
    over the whole-trace run (same subtraction constant here: the estimate is exact for this trace's first piece)."""
    from cusumtools_b200 import writer
    codes, _ = synth.c1_trace(n=2_000_000, n_events=300, seed=33)
    host = torch.from_numpy(codes).pin_memory()
    kw = dict(baseline_block=65536, cusum_delta=400.0, cusum_h=10.0, **KW)
    a = pipeline.TraceAnalyzer(len(codes), S, 1e5, 8, **kw)
    ra = a.run(host.cuda())
    ta = writer.event_table_from_result(a, ra, samplerate=synth.FS)
    b = pipeline.StreamingAnalyzer(len(codes), S, 1e5, 8, shards=4, **kw)
    rb = b.run_from_host(host)
    tb = writer.event_table_from_stream(b, rb, samplerate=synth.FS)
    assert list(tb.events) == list(ta.events) and list(tb.rate) == list(ta.rate)
    assert np.array_equal(tb.rate["id"], ta.rate["id"]) and np.array_equal(tb.rate["type"], ta.rate["type"])
    assert np.allclose(tb.rate["start_time_s"], ta.rate["start_time_s"], rtol=0, atol=1.01 / synth.FS)
    assert np.array_equal(tb.events["id"], ta.events["id"]) and np.array_equal(tb.events["n_levels"], ta.events["n_levels"])
    for col in ("effective_baseline_pA", "average_blockage_pA", "max_blockage_pA", "max_deviation_pA", "residual_pA"):
        close = np.isclose(tb.events[col], ta.events[col], rtol=1e-3, atol=0.5)
        assert np.mean(close) > 0.98, col          # (a boundary decision on a line may fall either way: see _tables_agree)


def test_config_c1_end_to_end_against_the_cpu_path():
    """BASELINE.json configs[0]: 1 s synthetic Chimera trace (4 166 666 samples), 8-pole 100 kHz Bessel,
    1000 injected two-level events, threshold detection + CUSUM+.  The GPU path runs on the codes; the CPU
    path is the reference's call sequence (scale_raw_data -> median pad -> scipy filtfilt, float64) followed
    by the oracle's detection / CUSUM+ on ITS OWN filtered trace.  End to end the two filtered traces differ
    by float32 rounding, so indices may move where a sample sits within that tolerance of a line (SURVEY.md
    H2): every injected event must be found by both, and event boundaries / changepoints must agree
    to within one sample on (almost) all of them."""
    from oracle import trace_oracle as to
    codes, true_starts = synth.c1_trace()
    n = len(codes)
    assert n == 4_166_666 and len(true_starts) == 1000
    an = pipeline.TraceAnalyzer(n, S, 1e5, 8, baseline_block=65536, cusum_delta=400.0, cusum_h=10.0, **KW)
    r = an.run(torch.from_numpy(codes).cuda())
    y_ref = to.filter_data(to.scale_raw_data(codes, S), synth.FS, 1e5, 8)
    assert np.abs(r.filtered.cpu().numpy() - y_ref).max() < 0.05
    ref = oracle_chain(y_ref.astype(np.float32), n, 65536)
    gs, ge = r.events.starts.cpu().numpy(), r.events.ends.cpu().numpy()
    assert len(gs) == len(ref["s"])
    assert 1000 <= len(gs) <= 1002                      # + at most the pad artefacts at the two ends
    assert np.abs(gs - ref["s"]).max() <= 1 and np.abs(ge - ref["e"]).max() <= 1
    assert np.mean(gs == ref["s"]) > 0.995 and np.mean(ge == ref["e"]) > 0.995
    ok = ref["ok"]
    gnl = r.levels.n_levels.cpu().numpy()[ok]
    assert np.mean(gnl == ref["lv"][0]) > 0.99
    same = gnl == ref["lv"][0]
    ged = r.levels.edges.cpu().numpy()[ok][same]
    assert np.mean(np.abs(ged - ref["lv"][1][same]).max(axis=1) <= 1) > 0.99
    gm = r.levels.mean.cpu().numpy()[ok][same]
    nl = ref["lv"][0][same]
    lvl_err = max(np.abs(gm[i, :nl[i]] - ref["lv"][2][same][i, :nl[i]]).max() for i in range(0, len(nl), 10))
    assert lvl_err < 1.0                                 # pA; a changepoint moved by one sample shifts a level mean slightly


def _exact_pair(codes):
    from cusumtools_b200 import filters
    srt = np.sort(codes & np.uint16(filters.chimera_bitmask(S)))
    return int(srt[(codes.size - 1) // 2]), int(srt[codes.size // 2])


def test_median_routes_drift_and_window_miss():
    """The three routes of the exact median inside TraceAnalyzer.run (plot-trace.py:319: np.pad(mode='median')):
    (a) the eight-code window tallied by the forward pass and verified on the device (ct_median_verify: no host round
        trip between the passes),
    (b) a drifting baseline: the estimate is uncertain (MedianPlan.se > 0.8), host loop,
    (c) a distribution whose SAMPLE median sits 40 codes below the true one: the device-side verification reports a
        miss and the step is redone the host-driven way.  Median, pad value and filtered trace are the exact ones."""
    from cusumtools_b200 import filters
    from oracle import trace_oracle as to
    n = 5_000_000
    base, _ = synth.c1_trace(n=n, n_events=600, seed=7)
    drift = (base.astype(np.int64) + 4 * (np.arange(n) * 3000 // n)).astype(np.uint16)       # +3000 code steps (7 nA) over the trace
    # (c): stride-4 sampling (n // 2^20 = 4) sees only positions 0, 4, 8, ...; they hold code A, the others mostly B = A + 40 steps
    A = int(_exact_pair(base)[0])
    tri = np.full(n, A + 160, dtype=np.uint16)
    tri[::4] = A
    tri[1::4][: n // 4 - 2] = A                        # A holds just under half of all samples: the median is B
    seen = []
    for name, codes in (("narrow", base), ("drift", drift), ("miss", tri)):
        raw = torch.from_numpy(codes).cuda()
        an = pipeline.TraceAnalyzer(n, S, 1e5, 8, baseline_block=65536, maxpoints=4000, **KW)
        r = an.run(raw)
        seen.append(an.last_median_route)
        assert r.median_codes == _exact_pair(codes), name
        assert r.pad_value == float(np.median(to.scale_raw_data(codes, S))), name
        want = filters.dequant_filtfilt(raw, S, 1e5, 8, median_codes=r.median_codes).cpu().numpy()
        assert np.abs(r.detect_trace.cpu().numpy() - want).max() < 0.02, name
    assert _exact_pair(tri) == (A + 160, A + 160)
    assert seen == ["device", "host", "host after a device miss"]


def test_device_side_pad_when_the_estimate_is_off_by_two_codes():
    """The sampled positions (every 4th sample of a 5 M-sample trace) sit two code steps higher than the rest, so the
    estimate is median + 2 steps: the eight-code window still holds the median, ct_median_verify leaves a NON-ZERO pad on
    the device and ct_filter_forward_ends_u16 re-runs the end groups with it.  Median, pad value and the trace ends (where
    the pad acts) must be the exact ones."""
    from cusumtools_b200 import filters
    from oracle import trace_oracle as to
    n = 5_000_000
    codes, _ = synth.c1_trace(n=n, n_events=600, seed=11)
    codes = codes.copy()
    codes[::4] += np.uint16(8)
    raw = torch.from_numpy(codes).cuda()
    for fused in (True, False):
        an = pipeline.TraceAnalyzer(n, S, 1e5, 8, baseline_block=65536, maxpoints=4000, fused_count=fused, **KW)
        r = an.run(raw)
        assert an.last_median_route == "device"
        assert r.median_codes == _exact_pair(codes)
        res = an.median_result.cpu().numpy()
        assert res[3] == 0 and res[2:3].view(np.float32)[0] != 0.0          # status ok, pad_x = median - estimate != 0
        assert r.pad_value == float(np.median(to.scale_raw_data(codes, S)))
        want = to.filter_data(to.scale_raw_data(codes, S), synth.FS, 1e5, 8)
        got = r.detect_trace.cpu().numpy()
        assert np.abs(got[:3000] - want[:3000]).max() < 0.05 and np.abs(got[-3000:] - want[-3000:]).max() < 0.05
        assert np.abs(got - want).max() < 0.05


def test_median_verify_entry_point_against_the_host_logic():
    """ct_median_verify (one device thread) == median.verify (numpy) on random window counts: found / window
    above the median / window below it, four and eight codes, odd and even totals."""
    import ctypes as C
    from cusumtools_b200 import _lib, median
    L = _lib.lib()
    rng = np.random.default_rng(3)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for trial in range(200):
        nb = 4 if trial % 2 else 8
        c = np.zeros(9, dtype=np.int64)
        c[:1 + nb] = rng.integers(0, 50, 1 + nb)
        above = int(rng.integers(0, 120))
        c[0] = int(rng.integers(0, 120))
        n = int(c.sum()) + above
        if n == 0:
            continue
        k1, k2 = (n - 1) // 2, n // 2
        lo, step, est = 4000 + 4 * int(rng.integers(0, 50)), 4, 4100.0
        plan = median.MedianPlan(n, k1, k2, step, 2, int(est), lo)
        want, _ = median.verify(plan, torch.from_numpy(c[:9].copy()))
        if nb == 4 and want is not None and max(want) >= lo + 4 * step:
            want = None                                         # the host logic always looks at eight codes
        dev = torch.from_numpy(c).cuda()
        res = torch.zeros(4, dtype=torch.int32, device="cuda")
        _lib.check(L.ct_median_verify(dev.data_ptr(), nb, k1, k2, lo, step, est, res.data_ptr(), st), "ct_median_verify")
        out = res.cpu().numpy()
        if want is None:
            assert out[3] in (1, 2) and out[3] == (1 if k1 < c[0] else 2) and out[0] == 0 and out[1] == 0
        else:
            assert out[3] == 0 and (int(out[0]), int(out[1])) == want
            assert out[2:3].view(np.float32)[0] == np.float32(0.5 * (want[0] + want[1]) - est)
    assert L.ct_median_verify(dev.data_ptr(), 9, 0, 0, 0, 4, 0.0, res.data_ptr(), st) != 0      # nbins out of range
