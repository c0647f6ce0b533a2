"""The float32-input path of the split filter (ct_filtfilt_f32: filters.bessel_filtfilt, bessel_lfilter,
bessel_filtfilt_odd) and the causal-only mode (forward pass straight to the output) of both input kinds, over the
configurations test_gpu_filter_grid.py covers for codes: every section count and scratch decimation, run lengths
R = 256 .. 4096, pads between 0 and the warm-up, unaligned input and output views, and trace lengths from 1 sample.

The float instantiation of the forward kernel is code of its own: two 32-sample stages per tile, a FLOAT32 tensor map,
a guarded fill with the pad value outside the data, x - pad instead of the integer subtract of the codes, and its own
host mapping of the pad and offset (no integer / fraction split of the pad).  Every output is checked against float64
scipy in cascade form (sosfiltfilt / sosfilt of bessel(..., output="sos")) computed from the float32 samples the
kernel read, within 0.05 pA and 1e-5 of the level, ends included; runs that differ only in the alignment of their
views must agree bit for bit.  Each case asserts the (sections, decimation, run length) it ran and whether its
pointers allowed the tensor maps (16-byte alignment)."""
import ctypes as C

import numpy as np
import pytest
import torch
from scipy.signal import bessel, sosfilt, sosfilt_zi, sosfiltfilt

from cusumtools_b200 import _lib, detect, filters, synth
from oracle import trace_oracle as to
from test_gpu_filter_grid import (ABS_TOL, DESIGNS, PAD, _design, check_samples, length_for_run, ragged_origin,
                                  run_length, sample_windows, stats_block)

pytestmark = pytest.mark.gpu
S = synth.CHIMERA_SETTINGS
S16 = dict(S, SETUP_ADCBITS=np.array([[16]]))            # every code is a code: two neighbours have a median of x.5
N_GRID = 1_234_567
N_SHORT = 300_001                                         # R = 256 for every design whose warm-up allows it
RUNS = (256, 512, 1024, 2048, 4096)
CAUSAL = {1: "1p_200k", 2: "4p_100k", 3: "5p_100k", 4: "8p_100k", 5: "9p_200k"}   # sections: design with Hw <= 256
ODD_N = 20_000_017                                        # runs of 512 with no pad


# ------------------------------------------------------------------------------------------------ helpers
def sos_of(poles, cutoff):
    return bessel(poles, 2.0 * cutoff / synth.FS, "low", output="sos")


def dequant(raw, settings=S):
    """Codes -> float32 pA on the device (ct_dequant_u16, the loader's path)."""
    out = torch.empty(raw.numel(), dtype=torch.float32, device=raw.device)
    alpha, beta = filters.chimera_affine(settings)
    rc = _lib.lib().ct_dequant_u16(raw.data_ptr(), raw.numel(), filters.chimera_bitmask(settings), alpha, beta,
                                   out.data_ptr(), filters._stream_ptr(out))
    _lib.check(rc, "ct_dequant_u16")
    return out


def host64(t):
    return t.cpu().numpy().astype(np.float64)


def filtfilt_ref(sos, x, pv, pad):
    """float64 filtfilt over np.pad(x, pad, constant=pv) with the forward pass starting from the steady state of pv
    and the backward pass from that of the last forward output: for pad > 0 exactly sosfiltfilt(padtype=None), for
    pad = 0 the same with pv in place of x[0] (the kernel's left end always settles on the pad value)."""
    xp = np.pad(x, pad, mode="constant", constant_values=pv)
    zi = sosfilt_zi(sos)
    f, _ = sosfilt(sos, xp, zi=zi * pv)
    b, _ = sosfilt(sos, f[::-1], zi=zi * f[-1])
    return b[::-1][pad:xp.size - pad]


def causal_ref(sos, x, v):
    return sosfilt(sos, x, zi=sosfilt_zi(sos) * v)[0]


def plan(design, n, pad, forward_only=False):
    """(sections, scratch decimation, run length) the library picks: the forward-only mode runs without a pad."""
    coef, H = filters.make_coef(design), filters.warmup_samples(design)
    L = _lib.lib()
    if forward_only:
        return coef.nsec, None, int(L.ct_filtfilt_stats_granule(n, 0, H)) // 64
    return coef.nsec, int(L.ct_filter_decimation(C.byref(coef), pad, H)), int(L.ct_filtfilt_stats_granule(n, pad, H)) // 64


def tma_ok(t):
    """The tensor maps of a trace or output need a 16-byte aligned start (run rows are multiples of 64 samples)."""
    return t.data_ptr() % 16 == 0


def view_at(src, offset, extra=1, fill=float("nan")):
    """A copy of `src` starting `offset` elements into a fresh buffer (with `fill` before and after it)."""
    buf = torch.full((src.numel() + offset + extra,), fill, dtype=src.dtype, device=src.device)
    v = buf[offset:offset + src.numel()]
    v.copy_(src)
    return buf, v


def out_at(n, offset, device="cuda"):
    buf = torch.full((n + offset + 1,), float("nan"), dtype=torch.float32, device=device)
    return buf, buf[offset:offset + n]


def check_untouched(buf, offset, n):
    """Nothing was written before or after the output view."""
    assert torch.isnan(buf[:offset]).all() and torch.isnan(buf[offset + n:]).all()


def fractional(v):
    """A float32 pad with a fractional part of about 0.37: a kernel that split it like the integer codes, or lost
    it, is off by more than the tolerance."""
    return float(np.float32(np.floor(v) + 37.37))


def check_windows_f32(x, y, starts, pv, sos, H, W=256):
    """Windows of the output against sosfiltfilt of the float32 input with 10 H samples of context; the constant pad
    only at the true trace ends."""
    n = x.numel()
    M = 10 * H
    for a in starts:
        lo, hi = max(0, a - M), min(n, a + W + M)
        xs = host64(x[lo:hi])
        left, right = (PAD if lo == 0 else 0), (PAD if hi == n else 0)
        xp = np.pad(xs, (left, right), mode="constant", constant_values=pv)
        want = sosfiltfilt(sos, xp, padtype=None)[left + a - lo:left + a - lo + W]
        check_samples(y[a:a + W].cpu().numpy(), want)


def test_cases_cover_every_section_count_decimation_and_run_length():
    every = {(s, D) for s in range(1, 6) for D in (1, 2, 4)} - {(1, 4)}
    assert {plan(_design(p, c)[0], N_GRID, PAD)[:2] for p, c, *_ in DESIGNS.values()} == every      # A
    d, _, H = _design(8, 1e5)
    assert {plan(d, length_for_run(R, H), PAD)[2] for R in RUNS} == set(RUNS)                        # B
    d20, _, H20 = _design(4, 2e4)
    assert H20 > 256 and plan(d20, length_for_run(1024, H20), PAD)[2] == 1024
    assert {plan(d, N_SHORT, PAD)[2], plan(d, length_for_run(1024, H), PAD)[2]} == {256, 1024}       # C
    for name in CAUSAL.values():                                                                     # E
        p, c, *_ = DESIGNS[name]
        assert plan(_design(p, c)[0], N_SHORT, 0, True)[2] == 256
    assert sorted(plan(_design(*DESIGNS[nm][:2])[0], N_SHORT, 0, True)[0] for nm in CAUSAL.values()) == [1, 2, 3, 4, 5]


# ------------------------------------------------------------------------------------------------ A: design grid
@pytest.fixture(scope="module")
def grid_samples():
    codes, _ = synth.c1_trace(n=N_GRID, n_events=(N_GRID - 4000) // synth.EVENT_PERIOD, seed=41)
    x = dequant(torch.from_numpy(codes).cuda())
    return x, host64(x)


def one_call_block_sums(x, poles, cutoff, pv, origin, block, bmin=4700.0, bmax=5300.0):
    """ct_filtfilt_f32 with fused baseline block sums; they must equal ct_block_stats_f32 on its output."""
    d, coef, H = _design(poles, cutoff)
    n = x.numel()
    L = _lib.lib()
    bl = detect.new_baseline(n - origin, block, bmin, bmax, x.device)
    st = detect.stats_args(bl, origin=origin)
    wsb = int(L.ct_filtfilt_workspace_bytes(n, PAD, H))
    ws = torch.empty(wsb, dtype=torch.uint8, device=x.device)
    y = torch.empty(n, dtype=torch.float32, device=x.device)
    rc = L.ct_filtfilt_f32(x.data_ptr(), n, PAD, float(pv), C.byref(coef), H, 0, y.data_ptr(), ws.data_ptr(), wsb,
                           C.byref(st), filters._stream_ptr(x))
    _lib.check(rc, "ct_filtfilt_f32")
    ref = detect.baseline_blocks(y[origin:], block, bmin, bmax)
    assert int(ref.dev["cnt"].sum()) > 0
    for k in ("cnt", "s1", "s2"):
        assert torch.equal(bl.dev[k], ref.dev[k]), k
    return y


@pytest.mark.parametrize("name", list(DESIGNS))
def test_float_input_per_design(grid_samples, name):
    poles, cutoff, nsec, D, R = DESIGNS[name]
    d, coef, H = _design(poles, cutoff)
    x, x64 = grid_samples
    assert plan(d, x.numel(), PAD) == (nsec, D, R) and tma_ok(x)
    sos = sos_of(poles, cutoff)
    y = filters.bessel_filtfilt(x, synth.FS, cutoff, poles)          # pad = the median of the samples
    med = filters.float_median(x)
    assert med == np.median(x64)
    check_samples(y.cpu().numpy(), filtfilt_ref(sos, x64, np.float32(med), PAD))
    pv = fractional(med)                                              # a pad with a fraction, 37 pA off the median
    y2 = filters.bessel_filtfilt(x, synth.FS, cutoff, poles, pad_value=pv)
    check_samples(y2.cpu().numpy(), filtfilt_ref(sos, x64, pv, PAD))
    G = 64 * R
    if name == "8p_100k":
        y0 = one_call_block_sums(x, poles, cutoff, pv, 0, stats_block(G))
        assert torch.equal(y0, y2)                                    # same run grid: the tally changes nothing
        y1 = one_call_block_sums(x, poles, cutoff, pv, ragged_origin(G), stats_block(G))
        check_samples(y1.cpu().numpy(), filtfilt_ref(sos, x64, pv, PAD))
    elif name == "10p_900k":
        y0 = one_call_block_sums(x, poles, cutoff, pv, 0, stats_block(G))
        assert torch.equal(y0, y2)


# -------------------------------------------------------------------------------------------- B: run lengths
@pytest.mark.parametrize("poles,cutoff,R", [(8, 1e5, R) for R in RUNS] + [(4, 2e4, 1024)])
def test_float_input_per_run_length(poles, cutoff, R):
    d, coef, H = _design(poles, cutoff)
    n = length_for_run(R, H)
    raw = synth.device_trace(n, "cuda", seed=1000 + R)
    x = dequant(raw)
    del raw
    nsec, D, R_got = plan(d, n, PAD)
    assert R_got == R and n % 64 and tma_ok(x)
    assert (nsec, D) == ((4, 4) if poles == 8 else (2, 4))
    y = filters.bessel_filtfilt(x, synth.FS, cutoff, poles)
    pv = np.float32(filters.float_median(x))
    G = 64 * R
    check_windows_f32(x, y, sample_windows(n, 0, R, G), pv, sos_of(poles, cutoff), H)
    del x, y
    torch.cuda.empty_cache()


# -------------------------------------------------------------------------------------------- C: alignment
ALIGN_CASES = [(1, 0), (2, 0), (3, 0), (0, 1), (1, 1), (3, 1)]          # (input offset, output offset) in floats


@pytest.mark.parametrize("R", [256, 1024])
def test_float_alignment_is_invisible(R):
    """Unaligned views take the guarded fill and the guarded stores everywhere: the same arithmetic, bit for bit."""
    d, coef, H = _design(8, 1e5)
    n = N_SHORT if R == 256 else length_for_run(R, H)
    assert plan(d, n, PAD) == (4, 4, R) and plan(d, n, 0, True)[2] == R
    x = dequant(synth.device_trace(n, "cuda", seed=77 + R))
    assert tma_ok(x)
    pv = fractional(filters.float_median(x))
    ya = filters.bessel_filtfilt(x, synth.FS, 1e5, 8, pad_value=pv)
    fa = filters.bessel_lfilter(x, synth.FS, 1e5, 8, initial=pv)
    for ki, ko in ALIGN_CASES:
        _, xv = view_at(x, ki)
        assert tma_ok(xv) == (ki == 0)
        for fn, want in ((filters.bessel_filtfilt, ya), (filters.bessel_lfilter, fa)):
            buf, ov = out_at(n, ko)
            assert tma_ok(ov) == (ko == 0)
            kw = dict(pad_value=pv) if fn is filters.bessel_filtfilt else dict(initial=pv)
            y = fn(xv, synth.FS, 1e5, 8, out=ov, **kw)
            assert y.data_ptr() == ov.data_ptr()
            assert torch.equal(y, want), (fn.__name__, ki, ko)
            check_untouched(buf, ko, n)
        del xv
    sos = sos_of(8, 1e5)
    if R == 256:
        x64 = host64(x)
        check_samples(ya.cpu().numpy(), filtfilt_ref(sos, x64, pv, PAD))
        check_samples(fa.cpu().numpy(), causal_ref(sos, x64, pv))
    else:
        check_windows_f32(x, ya, sample_windows(n, 0, R, 64 * R), pv, sos, H)
        k = 1 << 20                                  # the causal output's first million samples
        check_samples(fa[:k].cpu().numpy(), causal_ref(sos, host64(x[:k]), pv))


# -------------------------------------------------------------------------------------------- D: pads
@pytest.mark.parametrize("name", ["8p_100k", "8p_250k"])
def test_float_pads_below_the_warmup(name):
    poles, cutoff, _, D, _ = DESIGNS[name]
    d, coef, H = _design(poles, cutoff)
    Hw = -(-H // 64) * 64
    codes, _ = synth.c1_trace(n=N_SHORT, n_events=70, seed=8)
    x = dequant(torch.from_numpy(codes).cuda())
    x64 = host64(x)
    sos = sos_of(poles, cutoff)
    pv = fractional(filters.float_median(x))
    for pad, want_d in ((0, 1), (Hw - 64, 1), (1000, D)):
        assert plan(d, N_SHORT, pad) == (4, want_d, 256)
        y = filters.bessel_filtfilt(x, synth.FS, cutoff, poles, pad_value=pv, padding=pad)
        check_samples(y.cpu().numpy(), filtfilt_ref(sos, x64, pv, pad))


def odd_reference(x, poles, cutoff):
    """to.filter_data_edge in cascade form: edge pad by `poles`, odd extension of 3 (poles + 1) samples, filtfilt from
    the steady states of its first sample and of the last forward output, [poles:-poles]."""
    xe = np.pad(x, poles, mode="edge")
    return sosfiltfilt(sos_of(poles, cutoff), xe, padtype="odd", padlen=3 * (poles + 1))[poles:-poles]


@pytest.mark.parametrize("poles", [2, 4, 5, 8])
def test_float_odd_extension_at_long_runs(poles):
    d, coef, H = _design(poles, 1e5)
    raw = synth.device_trace(ODD_N, "cuda", seed=300 + poles)
    x = dequant(raw)
    del raw
    ext = ODD_N + 2 * poles + 6 * (poles + 1)            # what the kernel filters, without a pad
    assert plan(d, ext, 0) == (coef.nsec, 1, 512)
    y = filters.bessel_filtfilt_odd(x, synth.FS, 1e5, poles)
    assert y.shape == x.shape
    x64 = host64(x)
    head = x64[:50_000]                                  # the cascade restatement is the reference's own operation
    assert np.abs(odd_reference(head, poles, 1e5) - to.filter_data_edge(head, synth.FS, 1e5, poles)).max() < 1e-3
    check_samples(y.cpu().numpy(), odd_reference(x64, poles, 1e5))


# ------------------------------------------------------------------------------------- E: causal-only mode
@pytest.fixture(scope="module")
def causal_codes():
    """16-bit codes (mask 0xFFFF) long enough for runs of 1024 in the causal mode; R = 256 takes a prefix."""
    d, _, H = _design(8, 1e5)
    return synth.device_trace(length_for_run(1024, H), "cuda", seed=5, settings=S16)


@pytest.mark.parametrize("R", [256, 1024])
@pytest.mark.parametrize("nsec", sorted(CAUSAL))
def test_causal_mode_both_input_kinds(causal_codes, nsec, R):
    poles, cutoff, *_ = DESIGNS[CAUSAL[nsec]]
    d, coef, H = _design(poles, cutoff)
    raw = causal_codes if R == 1024 else causal_codes[:N_SHORT]
    n = raw.numel()
    assert plan(d, n, 0, True) == (nsec, None, R)
    sos = sos_of(poles, cutoff)
    codes = raw.cpu().numpy()

    # codes: the median of two neighbouring codes, so the pad (and the kernel's subtracted code) is x.5
    c1 = int(np.median(codes))
    med = (c1, c1 + 1)
    v = float(np.median(filters.scale_codes_host(np.array(med, dtype=np.uint16), S16)))
    ya = filters.dequant_filtfilt(raw, S16, cutoff, poles, forward_only=True, padding=0, median_codes=med)
    assert tma_ok(raw) and tma_ok(ya)
    check_samples(ya.cpu().numpy(), causal_ref(sos, to.scale_raw_data(codes, S16), v))
    _, rv = view_at(raw.view(torch.int16), 1, fill=0)
    for src, ko in ((rv, 0), (raw, 1), (rv, 1)):
        buf, ov = out_at(n, ko)
        assert (tma_ok(src), tma_ok(ov)) == (src is raw, ko == 0)
        y = filters.dequant_filtfilt(src, S16, cutoff, poles, forward_only=True, padding=0, median_codes=med, out=ov)
        assert torch.equal(y, ya), ko
        check_untouched(buf, ko, n)
    del rv

    # float samples with a fractional initial value
    x = dequant(raw, S16)
    x64 = host64(x)
    v = fractional(np.median(x64))
    fa = filters.bessel_lfilter(x, synth.FS, cutoff, poles, initial=v)
    assert tma_ok(x) and tma_ok(fa)
    check_samples(fa.cpu().numpy(), causal_ref(sos, x64, v))
    _, xv = view_at(x, 1)
    for src, ko in ((xv, 0), (x, 1), (xv, 1)):
        buf, ov = out_at(n, ko)
        assert (tma_ok(src), tma_ok(ov)) == (src is x, ko == 0)
        y = filters.bessel_lfilter(src, synth.FS, cutoff, poles, initial=v, out=ov)
        assert torch.equal(y, fa), ko
        check_untouched(buf, ko, n)


# ----------------------------------------------------------------------------- F: small and ragged lengths
@pytest.mark.parametrize("n", [1, 2, 17, 63, 64, 65, 511, 4097])
def test_float_ragged_lengths(n):
    poles, cutoff, nsec, D, _ = DESIGNS["8p_250k"]
    d, coef, H = _design(poles, cutoff)
    assert plan(d, n, PAD) == (nsec, D, 256) and plan(d, n, 0, True)[2] == 256
    codes, _ = synth.c1_trace(n=max(n, 3000), n_events=1, seed=n)
    x = dequant(torch.from_numpy(codes[:n].copy()).cuda())
    x64 = host64(x)
    sos = sos_of(poles, cutoff)
    y = filters.bessel_filtfilt(x, synth.FS, cutoff, poles)
    med = filters.float_median(x)
    assert med == np.median(x64)
    check_samples(y.cpu().numpy(), filtfilt_ref(sos, x64, np.float32(med), PAD))
    v = fractional(med)
    f = filters.bessel_lfilter(x, synth.FS, cutoff, poles, initial=v)
    check_samples(f.cpu().numpy(), causal_ref(sos, x64, v))


# ------------------------------------------------------------------------------------------- the out argument
def test_float_out_of_the_wrong_length_is_rejected():
    """Checked on the host before anything is launched: the buffers keep their contents."""
    x = dequant(torch.from_numpy(synth.c1_trace(n=5000, n_events=1, seed=3)[0]).cuda())
    for m in (4999, 5001, 0):
        out = torch.full((m,), 7.0, device="cuda")
        for kw in (dict(), dict(pad_value=5000.0), dict(forward_only=True, padding=0)):
            with pytest.raises(ValueError, match="wrong length"):
                filters.bessel_filtfilt(x, synth.FS, 1e5, 8, out=out, **kw)
        with pytest.raises(ValueError, match="wrong length"):
            filters.bessel_lfilter(x, synth.FS, 1e5, 8, out=out)
        torch.cuda.synchronize()
        assert bool((out == 7.0).all())
