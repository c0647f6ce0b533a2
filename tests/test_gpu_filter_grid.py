"""The split filter passes and the detector's chunk-extrema path over the configurations they are built for:
every section count 1-5, every scratch decimation D in {1, 2, 4}, odd numbers of warm-up tiles, and run lengths
R = 256 .. 4096 (the run grid of a long trace, G = 64 R samples per warp group).

The passes are driven through the C ABI with TraceAnalyzer.run's own call sequence (forward with the fused window
count, ct_median_verify, the end groups re-run with the device pad, backward with the fused block sums and chunk
extrema).  Every output is checked against a plain reference of the same operation:
  * samples: float64 scipy sosfiltfilt over the constant median pad (the reference's filter_data in cascade form),
    within 0.05 pA and 1e-5 of the level, ends included;
  * chunk extrema: torch min / max of the output, bit for bit;
  * block sums: ct_block_stats_f32 on the output, exact integers;
  * window count: a torch count of the masked codes, exact;
  * events / baseline table / CUSUM+ levels: the oracle chain on the analyzer's own output, bit for bit;
  * the detector's chunk-extrema pass: the detector without extrema and the C twin, on hand-built traces and extrema
    (ties with the lines, both signs, shifted arrays, widened extrema)."""
import ctypes as C

import numpy as np
import pytest
import torch
from scipy.signal import bessel, sosfiltfilt

from cusumtools_b200 import _lib, detect, filters, pipeline, synth
from cusumtools_b200.design import bessel_lowpass
from oracle import c_twin, events_oracle as eo, trace_oracle as to

pytestmark = pytest.mark.gpu
S = synth.CHIMERA_SETTINGS
PAD = 1000
ABS_TOL = 0.05
MASK = filters.chimera_bitmask(S)
STEP = 1 << (16 - int(np.squeeze(S["SETUP_ADCBITS"])))     # code step of a 14-bit ADC
N_GRID = 1_234_567                                         # design grid: R = 256 unless the warm-up forces more
KW = dict(threshold=5.0, hysteresis=1.0, cusum_delta=400.0, cusum_h=10.0)

# name: (poles, cutoff Hz, sections, scratch decimation D, run length R at N_GRID).  Warm-up tiles Hw / 64 in brackets;
# R is at least Hw, rounded up to a power of two.
DESIGNS = {
    "8p_100k": (8, 1e5, 4, 4, 256),        # [4]  the benchmark's design
    "8p_250k": (8, 2.5e5, 4, 2, 256),      # [2]
    "8p_900k": (8, 9e5, 4, 1, 256),        # [1]  the GUI default
    "8p_50k": (8, 5e4, 4, 4, 512),         # [8]
    "4p_100k": (4, 1e5, 2, 2, 256),        # [3]
    "5p_100k": (5, 1e5, 3, 2, 256),        # [3]  a first-order section
    "3p_200k": (3, 2e5, 2, 1, 256),        # [2]
    "10p_100k": (10, 1e5, 5, 4, 512),      # [5]
    "10p_900k": (10, 9e5, 5, 1, 256),      # [1]
    "2p_20k": (2, 2e4, 1, 2, 1024),        # [10] Hw = 640 forces R >= 1024 at any length
    "1p_200k": (1, 2e5, 1, 1, 256),        # [1]
    "4p_20k": (4, 2e4, 2, 4, 1024),        # [13]
    "5p_500k": (5, 5e5, 3, 1, 256),        # [1]
    "6p_75k": (6, 7.5e4, 3, 4, 512),       # [5]
    "9p_200k": (9, 2e5, 5, 2, 256),        # [3]
}


def _design(poles, cutoff):
    d = bessel_lowpass(poles, 2.0 * cutoff / synth.FS)
    return d, filters.make_coef(d), filters.warmup_samples(d)


def run_length(n, H):
    return int(_lib.lib().ct_filtfilt_stats_granule(int(n), PAD, int(H))) // 64


def length_for_run(R, H):
    """A ragged trace length (not a multiple of 64) at which the library picks runs of R samples: the shortest
    such length (bisection; the run length grows with the trace) plus a group and a half and a remainder."""
    lo, hi = 1, 1 << 40
    while lo < hi:
        mid = (lo + hi) // 2
        if run_length(mid, H) >= R:
            hi = mid
        else:
            lo = mid + 1
    G = 64 * R
    n = max(lo, 64 * G) + G + G // 2 + 4321
    while n % 64 == 0:
        n += 1
    assert run_length(n, H) == R, (R, n, run_length(n, H))
    return n


def masked_codes(raw):
    return raw.view(torch.int16).to(torch.int32) & MASK


def exact_median(masked):
    m = masked.numel()
    cdf = torch.bincount(masked, minlength=65536).cumsum(0)
    k = torch.tensor([(m - 1) // 2 + 1, m // 2 + 1], device=masked.device, dtype=cdf.dtype)
    c1, c2 = torch.searchsorted(cdf, k).tolist()
    return int(c1), int(c2)


def pad_value(c1, c2, settings=S):
    return float(np.median(filters.scale_codes_host(np.array([c1, c2], dtype=np.uint16), settings)))


def sos_reference(x, poles, cutoff, pv):
    """The reference's filter_data in cascade form: float64 sosfiltfilt over np.pad(x, 1000, constant=pv)."""
    sos = bessel(poles, 2.0 * cutoff / synth.FS, "low", output="sos")
    return sosfiltfilt(sos, np.pad(x, PAD, mode="constant", constant_values=pv), padtype=None)[PAD:-PAD]


def check_samples(got, want):
    err = np.abs(np.asarray(got, np.float64) - want)
    level = np.abs(want).max()
    assert err.max() <= ABS_TOL and err.max() <= 1e-5 * level, (float(err.max()), int(err.argmax()), float(level))


class Split:
    """One pass of the split filter the way TraceAnalyzer.run drives it."""

    def __init__(self, raw, design, *, origin, count_range, est, block, bmin=4700.0, bmax=5300.0, settings=S):
        L = _lib.lib()
        dev = raw.device
        n = raw.numel()
        coef, H = filters.make_coef(design), filters.warmup_samples(design)
        st = filters._stream_ptr(raw)
        wsb = int(L.ct_filtfilt_workspace_bytes(n, PAD, H))
        ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
        self.minmax = torch.full((2 * int(L.ct_filter_summary_count(n, PAD, H)),), float("nan"), device=dev)
        self.counts = torch.zeros(9, dtype=torch.int64, device=dev)
        self.median = torch.zeros(4, dtype=torch.int32, device=dev)       # CtMedianResult
        self.lo = int(est) - 3 * STEP
        cb, ce = count_range
        rc = L.ct_filter_forward_u16(raw.data_ptr(), n, PAD, float(est), MASK, 0.0, C.byref(coef), H, origin, 0, self.lo, STEP,
                                     cb, ce, self.counts.data_ptr(), 0, n, ws.data_ptr(), wsb, st)
        _lib.check(rc, "ct_filter_forward_u16")
        m = ce - cb
        rc = L.ct_median_verify(self.counts.data_ptr(), 8, (m - 1) // 2, m // 2, self.lo, STEP, float(est),
                                self.median.data_ptr(), st)
        _lib.check(rc, "ct_median_verify")
        rc = L.ct_filter_forward_ends_u16(raw.data_ptr(), n, PAD, float(est), MASK, self.median[2:].data_ptr(), C.byref(coef),
                                          H, origin, ws.data_ptr(), wsb, st)
        _lib.check(rc, "ct_filter_forward_ends_u16")
        self.bl = detect.new_baseline(n - origin, block, bmin, bmax, dev)
        stats = detect.stats_args(self.bl, origin=origin)
        alpha, _ = filters.chimera_affine(settings)
        offset = float(filters.scale_codes_host(np.array([est], dtype=np.uint16), settings)[0])
        self.y = torch.empty(n, dtype=torch.float32, device=dev)
        rc = L.ct_filter_backward(n, PAD, float(est), float(alpha), offset, C.byref(coef), H, origin, self.y.data_ptr(),
                                  ws.data_ptr(), wsb, C.byref(stats), self.minmax.data_ptr(), st)
        _lib.check(rc, "ct_filter_backward")
        torch.cuda.synchronize()
        self.origin, self.block, self.bmin, self.bmax = origin, block, bmin, bmax

    def check_median(self, c1, c2, est):
        r = self.median.cpu().numpy()
        pad_x = float(r[2:3].view(np.float32)[0])
        assert (int(r[0]), int(r[1]), int(r[3])) == (c1, c2, 0)
        assert pad_x == 0.5 * (c1 + c2) - est != 0.0          # the end groups really were re-run with a device pad

    def check_counts(self, masked, count_range):
        cb, ce = count_range
        m = masked[cb:ce]
        want = [int((m < self.lo).sum())] + [int((m == self.lo + i * STEP).sum()) for i in range(8)]
        assert self.counts.cpu().tolist() == want

    def check_chunk_extrema(self, G):
        """Entry c = (min, max) of y[64 c - s : 64 c - s + 64], s = (G - origin mod G) mod G, for every chunk inside [0, n)."""
        n = self.y.numel()
        s = (G - self.origin % G) % G
        nc = n // 64
        mm = self.minmax.view(-1, 2)
        assert s % 64 == 0 and s // 64 + nc <= mm.shape[0]
        ch = self.y[:64 * nc].view(nc, 64)
        got = mm[s // 64:s // 64 + nc]
        assert torch.equal(got[:, 0], ch.amin(1)), "chunk minima"
        assert torch.equal(got[:, 1], ch.amax(1)), "chunk maxima"

    def check_block_sums(self):
        ref = detect.baseline_blocks(self.y[self.origin:], self.block, self.bmin, self.bmax)
        assert int(ref.dev["cnt"].sum()) > 0
        for k in ("cnt", "s1", "s2"):
            assert torch.equal(self.bl.dev[k], ref.dev[k]), k


def check_one_call_block_sums(raw, poles, cutoff, median, origin, block, bmin=4700.0, bmax=5300.0):
    """The same fused sums through the one-call ct_filtfilt_u16."""
    bl = detect.new_baseline(raw.numel() - origin, block, bmin, bmax, raw.device)
    y = filters.dequant_filtfilt(raw, S, cutoff, poles, median_codes=median, stats=detect.stats_args(bl, origin=origin))
    ref = detect.baseline_blocks(y[origin:], block, bmin, bmax)
    for k in ("cnt", "s1", "s2"):
        assert torch.equal(bl.dev[k], ref.dev[k]), k
    return y


def stats_block(G):
    """The smallest baseline block the filter can tally: a whole number of groups, at least 65536 samples."""
    return G * max(1, -(-65536 // G))


def ragged_origin(G):
    return G + 64 * 37                    # a multiple of 64, not of G: the chunk-extrema shift is not 0


def ragged_count_range(n, G):
    return G // 2 + 3 * 64 + 5, n - G - 1001     # neither end on a group, run or 64-sample boundary


# ------------------------------------------------------------------------------------------------ A: design grid
@pytest.fixture(scope="module")
def grid_trace():
    codes, starts = synth.c1_trace(n=N_GRID, n_events=(N_GRID - 4000) // synth.EVENT_PERIOD, seed=41)
    return codes, starts


def test_grid_covers_every_section_count_decimation_and_odd_warmups():
    reached = set()
    odd = 0
    for poles, cutoff, nsec, D, R in DESIGNS.values():
        d, coef, H = _design(poles, cutoff)
        assert (coef.nsec, filters.scratch_decimation(d, PAD), run_length(N_GRID, H)) == (nsec, D, R)
        reached.add((nsec, D))
        tiles = -(-H // 64)
        odd += tiles > 1 and tiles % 2 == 1
    # every (sections, D) pair a Bessel design of order 1-10 can take; a single section never passes the D = 4 bound
    assert reached == {(s, D) for s in range(1, 6) for D in (1, 2, 4)} - {(1, 4)}
    assert odd >= 5


@pytest.mark.parametrize("name", list(DESIGNS))
def test_split_passes_per_design(grid_trace, name):
    poles, cutoff, nsec, D, R = DESIGNS[name]
    d, coef, H = _design(poles, cutoff)
    assert (coef.nsec, int(_lib.lib().ct_filter_decimation(C.byref(coef), PAD, H)), run_length(N_GRID, H)) == (nsec, D, R)
    codes, _ = grid_trace
    n = codes.size
    G = 64 * R
    raw = torch.from_numpy(codes).cuda()
    masked = masked_codes(raw)
    x = to.scale_raw_data(codes, S)
    block = stats_block(G)
    for origin, count_range in ((0, (0, n)), (ragged_origin(G), ragged_count_range(n, G))):
        c1, c2 = exact_median(masked[count_range[0]:count_range[1]])
        est = c1 + 2 * STEP                      # two code steps off: the device pad is not 0
        sp = Split(raw, d, origin=origin, count_range=count_range, est=est, block=block)
        sp.check_median(c1, c2, est)
        sp.check_counts(masked, count_range)
        sp.check_chunk_extrema(G)
        sp.check_block_sums()
        y = sp.y.cpu().numpy()
        check_samples(y, sos_reference(x, poles, cutoff, pad_value(c1, c2)))
        y1 = check_one_call_block_sums(raw, poles, cutoff, (c1, c2), origin, block)
        if poles == 8 and origin == 0:
            # the reference's own direct form: below Wn = 0.04 its DC gain is off (test_gpu_filter.py
            # test_scratch_decimation_branches); the allowance is that offset, computed exactly from its b, a
            from fractions import Fraction
            b, a = bessel(8, 2 * cutoff / synth.FS, "low")
            dc = float(sum(Fraction(float(v)) for v in b) / sum(Fraction(float(v)) for v in a))
            want = to.filter_data(x, synth.FS, cutoff, 8)
            bias = abs(dc * dc - 1.0) * np.abs(want).max()
            assert np.abs(y.astype(np.float64) - want).max() <= ABS_TOL + bias
            assert np.abs(y1.cpu().numpy().astype(np.float64) - want).max() <= ABS_TOL + bias


# -------------------------------------------------------------------------------------------- B: run lengths
@pytest.fixture(scope="module")
def long_trace():
    """Device traces at the ragged length of each run length (8 poles, 100 kHz), generated once per module."""
    H = filters.warmup_samples(bessel_lowpass(8, 2 * 1e5 / synth.FS))
    cache = {}

    def get(R):
        if R not in cache:
            cache[R] = synth.device_trace(length_for_run(R, H), "cuda", seed=R)
        return cache[R]
    yield get
    cache.clear()


def sample_windows(n, base, R, G, W=256):
    """Window starts at both trace ends and straddling run, group and baseline-block boundaries."""
    runs, groups = (n - base) // R, (n - base) // G
    b = [base + k * R for k in (1, 2, 63, 64, 65, runs // 2, runs - 1)]
    b += [base + k * G for k in (1, 2, groups // 2, groups)]
    b += [k << 20 for k in (1, max(1, (n >> 20) // 2), n >> 20)]
    starts = [0, n - W]
    for i, p in enumerate(b):
        for off in ((-3, 5) if i % 2 else (-7, 2)):
            starts.append(p + off - W // 2)
    return sorted({min(max(0, s), n - W) for s in starts})


def check_windows(raw, y, starts, pv, H, W=256):
    n = raw.numel()
    M = 10 * H
    sos = bessel(8, 2 * 1e5 / synth.FS, "low", output="sos")
    for a in starts:
        lo, hi = max(0, a - M), min(n, a + W + M)
        x = to.scale_raw_data(raw[lo:hi].cpu().numpy(), S)
        left, right = (PAD if lo == 0 else 0), (PAD if hi == n else 0)
        xp = np.pad(x, (left, right), mode="constant", constant_values=pv)
        want = sosfiltfilt(sos, xp, padtype=None)[left + a - lo:left + a - lo + W]
        check_samples(y[a:a + W].cpu().numpy(), want)


@pytest.mark.parametrize("R", [256, 512, 1024, 2048, 4096])
def test_split_passes_per_run_length(long_trace, R):
    raw = long_trace(R)
    n = raw.numel()
    d, coef, H = _design(8, 1e5)
    G = 64 * R
    assert int(_lib.lib().ct_filtfilt_stats_granule(n, PAD, H)) == G and n % 64
    assert (coef.nsec, filters.scratch_decimation(d, PAD)) == (4, 4)
    masked = masked_codes(raw)
    block = stats_block(G)
    for origin, count_range in ((0, (0, n)), (ragged_origin(G), ragged_count_range(n, G))):
        c1, c2 = exact_median(masked[count_range[0]:count_range[1]])
        est = c1 + 2 * STEP
        sp = Split(raw, d, origin=origin, count_range=count_range, est=est, block=block)
        sp.check_median(c1, c2, est)
        sp.check_counts(masked, count_range)
        sp.check_chunk_extrema(G)
        sp.check_block_sums()
        base = -((G - origin % G) % G)
        check_windows(raw, sp.y, sample_windows(n, base, R, G), pad_value(c1, c2), H)
        del sp
        check_one_call_block_sums(raw, 8, 1e5, (c1, c2), origin, block)
    del masked
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------ C: analyzer against the oracle chain
def oracle_chain(y, block, bmin, bmax, pad=100, minp=8, maxp=100000, delta=400.0, h=10.0, max_levels=16):
    """The oracle's stages 2-3 over the whole detection trace `y`, with the baseline window [bmin, bmax] and its centre
    c0 as new_baseline derives them."""
    c0 = np.float32(0.5 * (np.float32(bmin) + np.float32(bmax)))
    hw = max(float(c0) - float(np.float32(bmin)), float(np.float32(bmax)) - float(c0))
    sh = eo.stats_shift(hw, block)
    cnt, s1, s2 = c_twin.block_stats(y, block, bmin, bmax, c0, sh)
    mean, std = eo.baseline_from_stats(cnt, s1, s2, c0, sh)
    sign, ts, te = eo.thresholds(mean, std, 5.0, 1.0)
    s, e, o = c_twin.detect_events(y, block, sign, ts, te)
    w0, w1, typ = eo.event_windows(s, e, len(y), pad, minp, maxp)
    ok = typ == 0
    offs = np.concatenate(([0], np.cumsum((w1 - w0)[ok])))
    flat = np.concatenate([y[a:b] for a, b in zip(w0[ok], w1[ok])]) if ok.any() else np.zeros(0, np.float32)
    lv = c_twin.cusum_batch(flat, offs, delta, h, max_levels)
    return dict(mean=mean, std=std, sign=sign, ts=ts, te=te, s=s, e=e, o=o, w0=w0, w1=w1, typ=typ, ok=ok, lv=lv)


def check_against_chain(r, ref):
    assert np.array_equal(r.baseline.mean, ref["mean"]) and np.array_equal(r.baseline.std, ref["std"])
    assert np.array_equal(r.baseline.sign, ref["sign"])
    assert np.array_equal(r.baseline.t_start, ref["ts"]) and np.array_equal(r.baseline.t_end, ref["te"])
    assert np.array_equal(r.events.starts.cpu().numpy(), ref["s"])
    assert np.array_equal(r.events.ends.cpu().numpy(), ref["e"])
    assert r.events.open_start == ref["o"]
    assert np.array_equal(r.win_start.cpu().numpy(), ref["w0"]) and np.array_equal(r.win_end.cpu().numpy(), ref["w1"])
    assert np.array_equal(r.types.cpu().numpy(), ref["typ"])
    ok = ref["ok"]
    nl, ed, mu, sd, ov = ref["lv"]
    gnl = r.levels.n_levels.cpu().numpy()
    assert np.array_equal(gnl[ok], nl) and np.all(gnl[~ok] == 0)
    assert np.array_equal(r.levels.edges.cpu().numpy()[ok], ed)
    gm, gs = r.levels.mean.cpu().numpy()[ok], r.levels.std.cpu().numpy()[ok]
    for i in range(len(nl)):          # rows are only defined up to n_levels
        assert np.array_equal(gm[i, :nl[i]], mu[i, :nl[i]]) and np.array_equal(gs[i, :nl[i]], sd[i, :nl[i]])
    assert np.array_equal(r.levels.overflow.cpu().numpy()[ok], ov)


@pytest.mark.parametrize("name", list(DESIGNS))
def test_analyzer_matches_oracle_chain_per_design(grid_trace, name):
    poles, cutoff, _, _, R = DESIGNS[name]
    codes, starts = grid_trace
    raw = torch.from_numpy(codes).cuda()
    block = stats_block(64 * R)
    an = pipeline.TraceAnalyzer(codes.size, S, cutoff, poles, baseline_block=block, baseline_min=4700.0,
                                baseline_max=5300.0, **KW)
    assert an.fuse_stats
    r = an.run(raw)
    assert r.median_codes == exact_median(masked_codes(raw))
    y = r.detect_trace.cpu().numpy()
    ref = oracle_chain(y, block, 4700.0, 5300.0)
    check_against_chain(r, ref)
    assert len(starts) <= len(ref["s"]) + 2


def test_analyzer_matches_oracle_chain_at_the_benchmark_step_shape(long_trace):
    """R = 4096 (G = 262 144, 64 tiles per run) with 2^20-sample baseline blocks: the run grid and block size of
    the benchmark's step and of any trace longer than about 155 M samples on a B200."""
    raw = long_trace(4096)
    n = raw.numel()
    block = 1 << 20
    an = pipeline.TraceAnalyzer(n, S, 1e5, 8, baseline_block=block, baseline_min=4700.0, baseline_max=5300.0,
                                event_padding=100, minpoints=8, maxpoints=100_000, **KW)
    assert an.fuse_stats and filters.stats_granule(n, PAD, an.design) == 64 * 4096
    r = an.run(raw)
    assert r.median_codes == exact_median(masked_codes(raw))
    y = r.detect_trace.cpu().numpy()
    ref = oracle_chain(y, block, 4700.0, 5300.0)
    check_against_chain(r, ref)
    assert len(ref["s"]) > n // 5000


def negative_settings():
    """Settings under which pA = alpha (code - 32766): beta = -32766 alpha, so pA(65532 - code) = -pA(code) (to the
    rounding of the reference's scaling sequence)."""
    s = dict(S)
    vref = float(np.squeeze(S["SETUP_ADCVREF"]))
    gain = float(np.squeeze(S["SETUP_TIAgain"])) * float(np.squeeze(S["SETUP_preADCgain"]))
    s["SETUP_pAoffset"] = np.array([[vref / gain / 16384.0]])
    return s


def test_analyzer_matches_oracle_chain_on_a_negative_baseline(grid_trace):
    """The mirrored codes (code -> 65532 - code, still 14-bit codes) carry the negated current: a -5000 pA baseline
    with blockages toward zero.  Every block takes the negative-sign branch of the detector and its chunk extrema."""
    Sn = negative_settings()
    alpha, beta = filters.chimera_affine(Sn)
    assert abs(beta / alpha + 32766.0) < 1e-6
    codes, starts = grid_trace
    mirrored = (65532 - codes.astype(np.int64)).astype(np.uint16)
    assert np.all(mirrored & ~np.uint16(MASK) == 0)
    raw = torch.from_numpy(mirrored).cuda()
    block = 65536
    an = pipeline.TraceAnalyzer(mirrored.size, Sn, 1e5, 8, baseline_block=block, baseline_min=-5300.0,
                                baseline_max=-4700.0, **KW)
    assert an.fuse_stats
    r = an.run(raw)
    y = r.detect_trace.cpu().numpy()
    ref = oracle_chain(y, block, -5300.0, -4700.0)
    check_against_chain(r, ref)
    assert np.all(ref["sign"] == -1) and np.all(ref["mean"] < -4900)
    assert len(starts) <= len(ref["s"]) <= len(starts) + 2
    c1, c2 = r.median_codes
    check_samples(y, sos_reference(to.scale_raw_data(mirrored, Sn), 8, 1e5, pad_value(c1, c2, Sn)))


# ----------------------------------------------------------------- D: the detector's chunk-extrema path on its own
DET_BLOCK = 4096
G_MAX = 64 * 4096                         # the largest warp group of the filter: shifts up to G_MAX - 64


def detector_trace(n, seed):
    """Blocks of both signs with their own lines; events, samples between the lines, and samples and whole chunks
    exactly on the lines.  Built in the positive frame (baseline m, start line m - 50, end line m - 40) and
    multiplied by the block's sign."""
    rng = np.random.default_rng(seed)
    nb = (n + DET_BLOCK - 1) // DET_BLOCK
    sign = np.where(rng.random(nb) < 0.5, 1, -1).astype(np.int32)
    sign[0] = 1
    if nb > 1:
        sign[1] = -1
    m = (1000.0 + 400.0 * rng.random(nb)).astype(np.float32)
    tsp, tep = (m - np.float32(50)).astype(np.float32), (m - np.float32(40)).astype(np.float32)
    blk = np.arange(n) // DET_BLOCK
    v = (m[blk] + np.float32(20) * rng.random(n).astype(np.float32)).astype(np.float32)
    p = int(rng.integers(5, 40))
    while p < n:                          # events of 3..400 samples every 30..900 samples, the first one early
        q = min(n, p + int(rng.integers(3, 400)))
        v[p:q] = m[blk[p:q]] - np.float32(100) + np.float32(30) * rng.random(q - p).astype(np.float32)
        p = q + int(rng.integers(30, 900))
    k = rng.random(n)
    v[k < 0.02] = (m - np.float32(45))[blk[k < 0.02]]               # between the lines: no symbol
    v[(k >= 0.02) & (k < 0.03)] = tsp[blk[(k >= 0.02) & (k < 0.03)]]   # exactly on the start line: no symbol
    v[(k >= 0.03) & (k < 0.04)] = tep[blk[(k >= 0.03) & (k < 0.04)]]   # exactly on the end line: no symbol
    # whole chunks on the lines (position 64 j is a chunk start for the detector)
    for j in range(0, n // 64 - 2, 7):
        a = 64 * j
        t, e = tsp[blk[a]], tep[blk[a]]
        kind = (j // 7) % 6
        if kind == 0:                     # inside an event, then a chunk that starts ON the end line, then baseline
            v[a:a + 64] = m[blk[a]] - np.float32(100)
            v[a + 64] = e
            v[a + 65:a + 128] = m[blk[a]]
        elif kind == 1:                   # min == end line, everything else beyond it
            v[a:a + 64] = m[blk[a]]
            v[a + int(rng.integers(0, 64))] = e
        elif kind == 2:                   # max == start line, everything else inside
            v[a:a + 64] = m[blk[a]] - np.float32(100)
            v[a + int(rng.integers(0, 64))] = t
        elif kind == 3:                   # every sample on the start line
            v[a:a + 64] = t
        elif kind == 4:                   # min == start line, max == end line
            v[a:a + 64] = m[blk[a]] - np.float32(45)
            v[a + 3], v[a + 60] = t, e
        else:                             # a whole chunk on the end line after an event
            v[a - 10:a] = m[blk[a]] - np.float32(100)
            v[a:a + 64] = e
    y = (v * sign[blk]).astype(np.float32)
    ts, te = (tsp * sign).astype(np.float32), (tep * sign).astype(np.float32)
    bl = detect.Baseline(DET_BLOCK, mean=(m * sign).astype(np.float64), std=np.ones(nb), count=np.ones(nb, np.int64))
    bl.sign, bl.t_start, bl.t_end = sign, ts, te
    return y, bl


def chunk_extrema(y, sign, s, widen=None, seed=0):
    """The filter's chunk-extrema layout: entry c = (min, max) of y[64 c - s : 64 c - s + 64].  Entries of chunks that
    are not entirely inside [0, n) hold extrema that would make the chunk 'all beyond the start line' if they were
    read.  `widen`: push every min down and every max up by 1 ulp or by more (same events)."""
    n = y.size
    nc = n // 64
    E = (n + s) // 64 + 2
    blk = np.clip(np.arange(E) * 64 - s, 0, n - 1) // DET_BLOCK
    pos = np.asarray(sign)[blk] > 0
    mm = np.where(pos[:, None], np.float32(-1e30), np.float32(1e30)) * np.ones((E, 2), np.float32)
    if nc:
        ch = y[:64 * nc].reshape(nc, 64)
        lo, hi = ch.min(axis=1), ch.max(axis=1)
        if widen is not None:
            rng = np.random.default_rng(seed)
            big = rng.random(nc) < 0.3
            lo = np.where(big, lo - np.float32(widen), np.nextafter(lo, np.float32(-np.inf)))
            hi = np.where(big, hi + np.float32(widen), np.nextafter(hi, np.float32(np.inf)))
        mm[s // 64:s // 64 + nc, 0] = lo
        mm[s // 64:s // 64 + nc, 1] = hi
    return mm


@pytest.mark.parametrize("s", [0, 64, 4032, G_MAX - 64])
@pytest.mark.parametrize("n", [63, 64, 65, 4095, 4096, 4097, (1 << 20) + 13])
def test_detector_chunk_extrema_path(n, s):
    y, bl = detector_trace(n, seed=n + s)
    yt = torch.from_numpy(y).cuda()
    for state_in in (False, True):
        rs, re_, ro = c_twin.detect_events(y, DET_BLOCK, bl.sign, bl.t_start, bl.t_end, state_in=state_in)
        plain = detect.detect_events(yt, bl, state_in=state_in)
        assert plain.starts.tolist() == rs.tolist() and plain.ends.tolist() == re_.tolist() and plain.open_start == ro
        for widen in (None, 1.0, 300.0):
            mm = torch.from_numpy(chunk_extrema(y, bl.sign, s, widen, seed=n)).cuda()
            ev = detect.detect_events(yt, bl, state_in=state_in, chunk_minmax=mm.view(-1), minmax_shift=s)
            assert ev.starts.tolist() == rs.tolist(), (state_in, widen)
            assert ev.ends.tolist() == re_.tolist(), (state_in, widen)
            assert ev.open_start == ro, (state_in, widen)
    if n > 1 << 16:
        assert len(rs) > 500                   # the trace does exercise the detector
