"""The detector (csrc/ct_detect.cu) at the sizes one benchmark step runs, and past them, bit for bit.

One step of config C2 analyses 2,499,999,600 samples (past 2^31) and finds about 600 000 events.  The traces here come
from tests/detect_cases.py, whose witnesses (checked on the host by tests/test_detect_cases_host.py) show that each
case reaches the scan boundaries it is named for, and whose segment reference is exact at any length:
  * the single-CTA scan with per = 1, 2 and 3 groups a thread, a last group of one sample, and both pass-1 kernels;
  * sample indices past 2^31 and 2^32 in pass 1, the chunk extrema and pass 2;
  * the event capacity: counters past it, nothing written past it, and the growth of detect.detect_events;
  * ct_event_windows at 1.2 M events (past its grid cap), on time-shard ranges and a capacity below the count;
  * ct_intra_crossings_f32 past its grid cap, on windows clipped by the trace ends and past 2^31;
  * TraceAnalyzer over the benchmark step's trace against the C twin chain.
Outputs start from sentinels, so a row a kernel should write and does not, or writes and should not, is seen.  Each
case checks the free device memory first and is skipped when the card, shared with other work, has too little."""
import numpy as np
import pytest
import torch

import detect_cases as dc
from cusumtools_b200 import _lib, detect, pipeline, synth
from oracle import c_twin, events_oracle as eo

pytestmark = pytest.mark.gpu

SENT = -0x5EED
SHAPES = {1 << 28: (1024, 1), (1 << 28) + 1: (1025, 2), (1 << 29) + 1: (2049, 3),
          dc.C2_SAMPLES: (9537, 10), (1 << 32) + (1 << 20) + 13: (16389, 17)}


@pytest.fixture(autouse=True)
def free_between_cases(record_property):
    torch.cuda.reset_peak_memory_stats()
    yield
    torch.cuda.synchronize()
    record_property("max_memory_allocated_GB", round(torch.cuda.max_memory_allocated() / 1e9, 2))
    torch.cuda.empty_cache()


def need(nbytes: float):
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes:
        pytest.skip(f"needs {nbytes / 1e9:.1f} GB of free device memory, {free / 1e9:.1f} GB free")


def sms() -> int:
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def dev(a, dtype):
    return torch.from_numpy(np.ascontiguousarray(a, dtype)).cuda()


def stream():
    return torch.cuda.current_stream().cuda_stream


def chunk_minmax(y: torch.Tensor, shift: int) -> torch.Tensor:
    """(min, max) of every whole 64-sample chunk, entry c covering [64 c - shift, 64 c - shift + 64); the entries of
    chunks outside the data (the partial tail chunk among them) are NaN, which the kernel must never take as a verdict."""
    nfull = y.numel() // 64
    mm = torch.full((shift // 64 + nfull + 1, 2), float("nan"), dtype=torch.float32, device=y.device)
    v = y[:nfull * 64].view(-1, 64)
    step = 1 << 22
    for r0 in range(0, nfull, step):
        r1 = min(nfull, r0 + step)
        mm[shift // 64 + r0:shift // 64 + r1, 0] = v[r0:r1].amin(dim=1)
        mm[shift // 64 + r0:shift // 64 + r1, 1] = v[r0:r1].amax(dim=1)
    return mm


def detect_abi(c: dc.Case, y, mm, shift, capacity, extra=64):
    """ct_detect_f32 into sentinel-filled buffers of capacity + extra rows; returns (counts2, starts, ends) on the host."""
    L = _lib.lib()
    wsb = int(L.ct_detect_workspace_bytes(c.n))
    ws = torch.zeros(wsb, dtype=torch.uint8, device="cuda")
    starts = torch.full((capacity + extra,), SENT, dtype=torch.int64, device="cuda")
    ends = torch.full((capacity + extra,), SENT, dtype=torch.int64, device="cuda")
    counts = torch.full((2,), SENT, dtype=torch.int64, device="cuda")
    sg, ts, te = dev(c.sign, np.int32), dev(c.t_start, np.float32), dev(c.t_end, np.float32)
    rc = L.ct_detect_f32(y.data_ptr(), c.n, c.block, sg.data_ptr(), ts.data_ptr(), te.data_ptr(), int(c.state_in),
                         mm.data_ptr() if mm is not None else None, shift, ws.data_ptr(), wsb, starts.data_ptr(),
                         ends.data_ptr(), capacity, counts.data_ptr(), stream())
    _lib.check(rc, "ct_detect_f32")
    out = counts.cpu().numpy(), starts.cpu().numpy(), ends.cpu().numpy()
    del ws, starts, ends
    return out


def host_baseline(c: dc.Case) -> detect.Baseline:
    nb = c.sign.size
    bl = detect.Baseline(c.block, np.zeros(nb), np.ones(nb), np.ones(nb, np.int64))
    bl.sign, bl.t_start, bl.t_end = c.sign, c.t_start, c.t_end
    return bl


# ------------------------------------------------------------------------------------------- detection at scale
@pytest.mark.parametrize("variant", range(4), ids=["b4096", "b4096_in", "b2^20", "b2^20_in"])
@pytest.mark.parametrize("n", dc.SCAN_SIZES + dc.BIG_SIZES)
def test_detection_at_every_scan_boundary(n, variant):
    """Starts, ends, open_start and the counters of both pass-1 kernels (and the chunk extrema at two shifts) against
    the segment reference, on traces whose patterns sit on run, group, scan-range and block boundaries, on 2^31 and
    2^32, with a long event over a whole scan range, a quiet range outside any event and an event open at the end."""
    need(4.6 * n + 4e9)
    c = dc.scan_cases(n)[variant]
    assert (c.ng, c.per) == SHAPES[n]
    if n == (1 << 28) + 1:
        assert c.n - (c.ng - 1) * dc.GROUP_SAMPLES == 1                 # the last group holds one sample
    assert [k for k, v in c.witness.items() if not v] == []
    if n > 1 << 31:
        assert c.n - 1 >= 1 << 31 and "some_pattern_on_2^31" in c.witness
    if n > 1 << 32:
        assert c.n - 1 >= 1 << 32 and "some_pattern_on_2^32" in c.witness
    y = dc.materialise(c, "cuda", seed=variant)
    assert dc.symbols_match(c, y)
    rs, re = dc.reference_raw(c)
    want = dc.events_form(rs, re, c.state_in)
    cap = max(rs.size, re.size) + 16
    for shift in (None, 0, 192):
        mm = chunk_minmax(y, shift) if shift is not None else None
        counts, s, e = detect_abi(c, y, mm, shift or 0, cap)
        del mm
        assert counts.tolist() == [rs.size, re.size], shift
        assert np.array_equal(s[:rs.size], rs) and np.all(s[rs.size:] == SENT), shift
        assert np.array_equal(e[:re.size], re) and np.all(e[re.size:] == SENT), shift
        got = dc.events_form(s[:rs.size], e[:re.size], c.state_in)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]) and got[2] == want[2], shift
    # a capacity below the event count: the counters still count everything, nothing is written at or past capacity
    for capacity in (1, rs.size // 2):
        counts, s, e = detect_abi(c, y, None, 0, capacity)
        assert counts.tolist() == [rs.size, re.size]
        assert np.array_equal(s[:min(capacity, rs.size)], rs[:capacity]) and np.all(s[capacity:] == SENT)
        assert np.array_equal(e[:min(capacity, re.size)], re[:capacity]) and np.all(e[capacity:] == SENT)
    ev = detect.detect_events(y, host_baseline(c), state_in=c.state_in, capacity=3)    # grows and redoes
    assert np.array_equal(ev.starts.cpu().numpy(), want[0]) and np.array_equal(ev.ends.cpu().numpy(), want[1])
    assert ev.open_start == want[2]


# ------------------------------------------------------------------------------------------------ event windows
def window_events(E: int, n_total: int, seed: int = 7):
    """E sorted events over an n_total-sample trace, past 2^31: every type (0, 2, 3, 4), the first window before sample
    0, the last past n_total, and the event at E // 3 padded into its predecessor."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(8, 1500, E)
    lens[::4999] = 150_000                                      # type 3 (maxpoints 100 000)
    lens[3::1000] = rng.integers(1, 8, lens[3::1000].size)      # type 2 (minpoints 8)
    gaps = rng.integers(150, 2100, E)
    gaps[5::777] = rng.integers(1, 150, gaps[5::777].size)      # type 4: padding of 100 reaches a neighbour
    gaps[E // 3] = 40
    gaps[0] = 50                                                # the first window starts at -50
    ends = np.cumsum(gaps + lens).astype(np.int64)
    starts = ends - lens
    assert ends[-2] < n_total - 600
    starts[-1], ends[-1] = n_total - 500, n_total - 30           # the last window ends past n_total
    return starts, ends


@pytest.mark.parametrize("open_event", [False, True], ids=["ns_eq_ne", "open"])
def test_event_windows_past_the_grid_cap(open_event):
    """ct_event_windows on 1.2 M events with indices past 2^31 against eo.event_windows over the whole list, sliced to
    each time-shard range: the whole trace, a range whose bounds are event starts in the middle of the list, an
    empty range, a range past n_total and a capacity below the event count."""
    need(2e9)
    E, n, pad, minp, maxp = 1_200_000, dc.C2_SAMPLES, 100, 8, 100_000
    starts, ends = window_events(E, n)
    grid_rows = sms() * 8 * 256
    assert E > 3 * grid_rows and starts.max() > 1 << 31
    ns = E + 1 if open_event else E
    st_h = np.append(starts, n - 10) if open_event else starts
    s_d, e_d = dev(st_h, np.int64), dev(ends, np.int64)
    counts = dev([ns, E], np.int64)
    L = _lib.lib()
    cases = [("whole", 0, n, E), ("mid", int(starts[E // 3]), int(starts[2 * E // 3]), E),
             ("empty", int(starts[100]) + 1, int(starts[101]), E), ("past_n", int(starts[E - 1000]), n + 10 ** 9, E),
             ("capacity", 0, n, E - 4321)]
    for name, lo, hi, capacity in cases:
        m = min(ns, E, capacity)
        w0r, w1r, tr = eo.event_windows(starts[:m], ends[:m], n, pad, minp, maxp)
        i0, i1 = np.searchsorted(starts[:m], lo), np.searchsorted(starts[:m], hi)
        if name == "whole":
            assert set(np.unique(tr).tolist()) == {0, 2, 3, 4} and w0r[0] < 0 and w1r[-1] > n
        if name == "mid":
            assert i0 > 0 and starts[i0] == lo and w0r[i0] < ends[i0 - 1] and i1 - i0 > grid_rows
        if name == "empty":
            assert i0 == i1
        w0 = torch.full((capacity + 64,), SENT, dtype=torch.int64, device="cuda")
        w1 = torch.full((capacity + 64,), SENT, dtype=torch.int64, device="cuda")
        ty = torch.full((capacity + 64,), SENT, dtype=torch.int32, device="cuda")
        out2 = torch.full((2,), SENT, dtype=torch.int64, device="cuda")
        rc = L.ct_event_windows(s_d.data_ptr(), e_d.data_ptr(), counts.data_ptr(), capacity, n, lo, hi, pad, minp, maxp,
                                w0.data_ptr(), w1.data_ptr(), ty.data_ptr(), out2.data_ptr(), stream())
        _lib.check(rc, "ct_event_windows")
        k = i1 - i0
        g0, g1, gt, o2 = w0.cpu().numpy(), w1.cpu().numpy(), ty.cpu().numpy(), out2.cpu().numpy()
        assert o2.tolist() == [k, i0], name
        assert np.array_equal(g0[:k], w0r[i0:i1]) and np.array_equal(g1[:k], w1r[i0:i1]), name
        assert np.array_equal(gt[:k], tr[i0:i1]), name
        assert np.all(g0[k:] == SENT) and np.all(g1[k:] == SENT) and np.all(gt[k:] == SENT), name


# ------------------------------------------------------------------------------------------- intra-event crossings
def intra_windows(c: dc.Case, E: int, seed: int = 3):
    """E windows over the case's trace: around its segment boundaries (so that they hold crossings), clipped at 0 and
    at n, past 2^31, and a few whose event start lies in the last block or past n_total; shuffled."""
    rng = np.random.default_rng(seed)
    n = c.n
    centres = rng.choice(c.seg_start[1:], E)
    half = rng.integers(1, 3000, E)
    w0 = centres - half
    w1 = centres + rng.integers(1, 3000, E)
    es = np.maximum(w0 + rng.integers(0, 200, E), 0)
    k = E // 20
    w0[:k] = -rng.integers(1, 400, k)                            # clipped at 0; the trace begins with crossings
    w1[:k] = rng.integers(100, 4000, k)
    w0[k:2 * k] = n - rng.integers(10, 3000, k)                  # clipped at n: the event open at n - 1 closes there
    w1[k:2 * k] = n + rng.integers(1, 500, k)
    es[k:2 * k] = np.where(np.arange(k) % 2 == 0, n - 100, n + 5000)     # last block; past n_total (clamped)
    order = rng.permutation(E)
    return w0[order], w1[order], es[order]


def intra_reference(yd, n, w0, w1, es, block, sign, ts, te):
    """eo.detect_events over the clipped window with the lines of the event start's block (clamped to the trace),
    an open crossing closed at the clipped end, indices relative to the unclipped window start."""
    a, b = max(int(w0), 0), min(int(w1), n)
    x = yd[a:b].cpu().numpy() if b > a else np.zeros(0, np.float32)
    kb = min(max(int(es) // block, 0), sign.size - 1)
    s, e, o = eo.detect_events(x, max(1, x.size), sign[kb:kb + 1], ts[kb:kb + 1], te[kb:kb + 1])
    if o >= 0:
        s, e = np.append(s, o), np.append(e, x.size)
    return np.stack((s, e), axis=1) + (a - int(w0)) if s.size else np.zeros((0, 2), np.int64)


def assert_intra_rows(cnt, pairs, rows, want_of, K):
    for i in rows:
        want = want_of(i)
        assert cnt[i] == len(want), i
        row = np.full(2 * K, SENT, np.int64)
        k = min(len(want), K)
        row[:2 * k] = want[:k].reshape(-1)
        assert np.array_equal(pairs[i], row), i


def subset_rows(w0, w1, n, nev):
    """The rows a scale test compares: the last grid-stride sweep, every row past 2^31, every clipped row, every 97th."""
    nw = sms() * 8 * 8
    last = (nev - 1) // nw * nw
    rows = np.arange(nev)
    sel = (rows >= last) | (w1[:nev] > 1 << 31) | (w0[:nev] < 0) | (w1[:nev] > n) | (rows % 97 == 0)
    return rows[sel], last


@pytest.mark.parametrize("K,short", [(1, 0), (8, 777)], ids=["K1", "K8_nev_dev"])
def test_intra_crossings_past_the_grid_cap(K, short):
    need(4.6 * dc.C2_SAMPLES + 4e9)
    n = dc.C2_SAMPLES
    c = dc.scale_case(n, 1 << 20, False, variant=2, extra={**dc.big_points(n), "head": [40, 300, 2000], "tail": [n - 200],
                                                               "burst": [(1 << 31) + 10_000 + 24 * j for j in range(12)]})
    assert [k for k, v in c.witness.items() if not v] == []
    y = dc.materialise(c, "cuda", seed=5)
    E = 30_000
    w0, w1, es = intra_windows(c, E)
    nw = sms() * 8 * 8
    assert E > 3 * nw and (w0 < 0).any() and (w1 > n).any() and (w0 > 1 << 31).any() and (es >= n).any()
    nev = E - short
    count = torch.full((E,), SENT, dtype=torch.int32, device="cuda")
    pairs = torch.full((E, 2 * K), SENT, dtype=torch.int32, device="cuda")
    nd = torch.tensor([nev], dtype=torch.int64, device="cuda") if short else None
    sg, ts, te = dev(c.sign, np.int32), dev(c.t_start, np.float32), dev(c.t_end, np.float32)
    w0d, w1d, esd = dev(w0, np.int64), dev(w1, np.int64), dev(es, np.int64)
    rc = _lib.lib().ct_intra_crossings_f32(y.data_ptr(), n, w0d.data_ptr(), w1d.data_ptr(), esd.data_ptr(), E,
                                           nd.data_ptr() if nd is not None else None, c.block, c.sign.size, sg.data_ptr(),
                                           ts.data_ptr(), te.data_ptr(), K, count.data_ptr(), pairs.data_ptr(), stream())
    _lib.check(rc, "ct_intra_crossings_f32")
    cnt, pr = count.cpu().numpy(), pairs.cpu().numpy().astype(np.int64)
    assert np.all(cnt[:nev] >= 0) and np.all(cnt[nev:] == SENT) and np.all(pr[nev:] == SENT)
    rows, last = subset_rows(w0, w1, n, nev)
    assert last > 0 and ((w0[rows] < 0) & (cnt[rows] > 0)).any() and ((w1[rows] > n) & (cnt[rows] > 0)).any()
    assert ((w0[rows] > 1 << 31) & (cnt[rows] > 0)).any() and (cnt[rows] > K).any()
    assert_intra_rows(cnt, pr, rows, lambda i: intra_reference(y, n, w0[i], w1[i], es[i], c.block, c.sign, c.t_start,
                                                               c.t_end), K)


# ------------------------------------------------------------------------------------ the analyzer at one step
def test_analyzer_at_the_benchmark_step():
    """TraceAnalyzer on the benchmark step's trace (bench.py, config C2) with intra-event crossings on: the baseline
    table, the lines, every event, window and type against the C twin chain over the detection trace, and the CUSUM+
    levels and crossings on the subset rows."""
    need(32e9)
    n = dc.C2_SAMPLES
    S = synth.CHIMERA_SETTINGS
    block, pad, minp, maxp, delta, h = 1 << 20, 100, 8, 100_000, 400.0, 10.0
    raw = synth.device_trace(n, torch.device("cuda"), seed=1234)
    an = pipeline.TraceAnalyzer(n, S, 100_000.0, 8, threshold=5.0, hysteresis=1.0, baseline_block=block,
                                baseline_min=4700.0, baseline_max=5300.0, event_padding=pad, minpoints=minp,
                                maxpoints=maxp, cusum_delta=delta, cusum_h=h, intra_threshold=50.0, intra_hysteresis=5.0)
    r = an.run(raw)
    del raw
    yh = r.detect_trace.cpu().numpy()
    c0 = np.float32(5000.0)
    sh = eo.stats_shift(300.0, block)
    cnt, s1, s2 = c_twin.block_stats(yh, block, 4700.0, 5300.0, c0, sh)
    mean, std = eo.baseline_from_stats(cnt, s1, s2, c0, sh)
    sign, ts, te = eo.thresholds(mean, std, 5.0, 1.0)
    assert np.array_equal(r.baseline.count, cnt)
    assert np.array_equal(r.baseline.mean, mean) and np.array_equal(r.baseline.std, std)
    assert np.array_equal(r.baseline.sign, sign)
    assert np.array_equal(r.baseline.t_start, ts) and np.array_equal(r.baseline.t_end, te)
    s, e, o = c_twin.detect_events(yh, block, sign, ts, te, cap=4_000_000)
    assert s.size > 9472 and s.max() > 1 << 31
    assert np.array_equal(r.events.starts.cpu().numpy(), s) and np.array_equal(r.events.ends.cpu().numpy(), e)
    assert r.events.open_start == o
    w0, w1, typ = eo.event_windows(s, e, n, pad, minp, maxp)
    assert np.array_equal(r.win_start.cpu().numpy(), w0) and np.array_equal(r.win_end.cpu().numpy(), w1)
    assert np.array_equal(r.types.cpu().numpy(), typ)
    rows, _ = subset_rows(w0, w1, n, s.size)
    lv = r.levels
    gnl, ged, gmu, gsd, gov = (t.cpu().numpy()[rows] for t in (lv.n_levels, lv.edges, lv.mean, lv.std, lv.overflow))
    ok = typ[rows] == 0
    assert ok.any() and np.all(gnl[~ok] == 0)
    okr = rows[ok]
    offs = np.concatenate(([0], np.cumsum(w1[okr] - w0[okr])))
    flat = np.concatenate([yh[w0[i]:w1[i]] for i in okr])
    nl, ed, mu, sd, ov = c_twin.cusum_batch(flat, offs, delta, h, lv.max_levels)
    assert np.array_equal(gnl[ok], nl) and np.array_equal(ged[ok], ed) and np.array_equal(gov[ok], ov)
    used = np.arange(lv.max_levels)[None, :] < nl[:, None]
    assert np.array_equal(gmu[ok][used], mu[used]) and np.array_equal(gsd[ok][used], sd[used])
    icnt, ipairs = r.intra[0].cpu().numpy(), r.intra[1].cpu().numpy()
    K = an.max_crossings
    for i in rows:
        kb = min(max((w0[i] + pad) // block, 0), mean.size - 1)
        a, b = max(w0[i], 0), min(w1[i], n)
        want = eo.intra_crossings(yh[a:b], mean[kb], std[kb], 50.0, 5.0) + (a - w0[i])
        assert icnt[i] == len(want), i
        k = min(len(want), K)
        assert np.array_equal(ipairs[i, :2 * k].reshape(-1, 2), want[:k]), i
    assert (icnt[rows] > 0).any()
