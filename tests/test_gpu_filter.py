"""GPU parity: fused dequantise + median-pad + Bessel filtfilt kernel vs the CPU oracle
(the reference's own call sequence) and vs fixtures produced by the reference itself.

Tolerances (SURVEY.md Appendix B.3, float32 state with median subtraction, Wn >= 0.04):
  |gpu - ref| <= 0.05 pA  and  <= 1e-5 of the baseline level.
The reference's float64 direct form has its own rounding-noise floor of ~3e-4 pA."""
import os

import numpy as np
import pytest
import torch
from scipy.signal import bessel, lfilter, lfilter_zi

from cusumtools_b200 import filters, median, synth
from cusumtools_b200.design import bessel_lowpass
from oracle import trace_oracle as to

pytestmark = pytest.mark.gpu
ABS_TOL = 0.05
S = synth.CHIMERA_SETTINGS


def gpu_filter(codes, cutoff, order, **kw):
    raw = torch.from_numpy(codes).cuda()
    y = filters.dequant_filtfilt(raw, S, cutoff, order, **kw)
    torch.cuda.synchronize()
    return y.cpu().numpy()


def check(got, want):
    err = np.abs(got.astype(np.float64) - want)
    assert err.max() <= ABS_TOL, err.max()
    assert err.max() <= 1e-5 * np.abs(want).max(), err.max()


def test_c1_slice_matches_oracle():
    codes, _ = synth.c1_trace(n=400000, n_events=95, seed=0)
    want = to.filter_data(to.scale_raw_data(codes, S), synth.FS, 1e5, 8)
    check(gpu_filter(codes, 1e5, 8), want)


@pytest.mark.parametrize("key", ["filt_100000_8", "filt_250000_8", "filt_900000_8", "filt_100000_4", "filt_200000_5"])
def test_reference_fixture(golden_dir, key):
    z = np.load(os.path.join(golden_dir, "filter_fixture.npz"))
    _, cutoff, order = key.split("_")
    check(gpu_filter(z["codes"], float(cutoff), int(order)), z[key])


def test_reference_fixture_even_length(golden_dir):
    z = np.load(os.path.join(golden_dir, "filter_fixture.npz"))
    check(gpu_filter(z["codes"][:-1].copy(), 1e5, 8), z["filt_even_100000_8"])


@pytest.mark.parametrize("n", [1, 2, 17, 511, 512, 513, 1000, 4095, 4096, 4097, 9000])
def test_ragged_lengths(n):
    codes, _ = synth.c1_trace(n=max(n, 3000), n_events=1, seed=n)
    codes = codes[:n].copy()
    want = to.filter_data(to.scale_raw_data(codes, S), synth.FS, 2.5e5, 8)
    check(gpu_filter(codes, 2.5e5, 8), want)


def test_empty_trace_is_rejected():
    raw = torch.zeros(0, dtype=torch.uint16, device="cuda")
    with pytest.raises(ValueError):
        filters.dequant_filtfilt(raw, S, 1e5, 8)


def test_unaligned_views():
    codes, _ = synth.c1_trace(n=70001, n_events=15, seed=3)
    raw = torch.from_numpy(codes).cuda()
    view = raw[1:]                       # 2-byte offset: vector loads are not possible
    out = torch.empty(70001, dtype=torch.float32, device="cuda")[1:]
    y = filters.dequant_filtfilt(view, S, 1e5, 8, out=out)
    torch.cuda.synchronize()
    want = to.filter_data(to.scale_raw_data(codes[1:], S), synth.FS, 1e5, 8)
    check(y.cpu().numpy(), want)


def test_run_length_is_invisible():
    """Runs are filtered independently with an Hw-sample warm-up, and the run length follows the trace
    length (256 for short traces, 4096 for long ones): the same samples embedded in a trace long enough for
    runs of 2048 samples or more must come out as they do in short traces (away from the ends)."""
    from cusumtools_b200 import _lib
    H = filters.warmup_samples(bessel_lowpass(8, 2 * 1e5 / synth.FS))

    def run(n):
        return int(_lib.lib().ct_filtfilt_stats_granule(n, 1000, H)) // 64

    lo, hi = 1, 1 << 40                  # the shortest trace with runs of 2048 samples (the run length grows with n)
    while lo < hi:
        mid = (lo + hi) // 2
        lo, hi = (lo, mid) if run(mid) >= 2048 else (mid + 1, hi)
    codes, _ = synth.c1_trace(n=6_000_000, n_events=1400, seed=9)
    raw = synth.device_trace(lo + 12_345, "cuda", seed=9)
    raw[:codes.size] = torch.from_numpy(codes).cuda()
    med = (40800, 40800)                 # one pad value for all lengths (the median of a prefix is not the trace's)
    full = filters.dequant_filtfilt(raw, S, 1e5, 8, median_codes=med)
    assert run(raw.numel()) >= 2048
    for n in (300_000, 1_500_000, 6_000_000):
        assert run(n) < run(raw.numel())
        part = gpu_filter(codes[:n].copy(), 1e5, 8, median_codes=med)
        assert np.abs(part[:n - 5000] - full[:n - 5000].cpu().numpy()).max() < 0.02


@pytest.mark.parametrize("cutoff,want_d", [(5e4, 4), (1e5, 4), (2.5e5, 2), (4e5, 2), (9e5, 1)])
def test_scratch_decimation_branches(cutoff, want_d):
    """The forward output crosses HBM at 1/4, 1/2 or full rate depending on the cascade's own stop band; every
    branch meets the same tolerance against the reference's float64 filtfilt (incl. the GUI default, 900 kHz)."""
    d = bessel_lowpass(8, 2 * cutoff / synth.FS)
    assert filters.scratch_decimation(d, 1000) == want_d
    assert filters.scratch_decimation(d, 0) == 1          # no settled pad: full rate
    codes, _ = synth.c1_trace(n=1_200_000, n_events=290, seed=17)
    want = to.filter_data(to.scale_raw_data(codes, S), synth.FS, cutoff, 8)
    got = gpu_filter(codes, cutoff, 8)
    # Below Wn = 0.04 the REFERENCE's float64 direct form loses its unit DC gain (the 9-tap denominator sums to ~1e-9
    # from coefficients of size ~70: at 50 kHz the exact DC gain of scipy's own b, a is 1 + 9.6e-6 per pass, i.e. the
    # reference reads +0.106 pA high on a 5 nA baseline).  The cascade here filters the median-subtracted signal with
    # DC gain 1, so the comparison allows for the reference's offset, computed exactly from its coefficients.
    from fractions import Fraction
    b, a = bessel(8, 2 * cutoff / synth.FS, "low")
    dc = float(sum(Fraction(float(v)) for v in b) / sum(Fraction(float(v)) for v in a))
    ref_bias = abs(dc * dc - 1.0) * np.abs(want).max()
    err = np.abs(got.astype(np.float64) - want)
    assert err.max() <= ABS_TOL + ref_bias, (err.max(), ref_bias)
    if ref_bias < 1e-3:
        check(got, want)


@pytest.mark.parametrize("poles", [2, 4, 8])
def test_odd_extension_mode_reference_fixture(golden_dir, poles):
    """The same mode against outputs of the reference's own App.filter_data (tests/golden/edge_fixture.npz)."""
    z = np.load(os.path.join(golden_dir, "edge_fixture.npz"))
    fs, fc = 1e3 * float(z["fs_khz"]), 1e3 * float(z["fc_khz"])
    for key in ("step", "noisy"):
        got = filters.bessel_filtfilt_odd(torch.from_numpy(z[key].astype(np.float32)).cuda(), fs, fc, poles).cpu().numpy()
        assert got.shape == z[key].shape
        assert np.abs(got - z[f"{key}_{poles}"]).max() <= 2e-6


@pytest.mark.parametrize("poles", [2, 4, 8])
def test_odd_extension_mode(poles):
    """legacy/bessel-filter.py:124-131: edge pad by `poles`, scipy's default filtfilt (odd extension of
    3*(poles+1) samples), then [poles:-poles]; on the reference's own 26-sample step and on a longer trace."""
    step = np.concatenate((np.zeros(13), np.ones(13)))
    codes, _ = synth.c1_trace(n=50000, n_events=10, seed=5)
    for x, fs, fc in ((step, 1.0, 0.1), (to.scale_raw_data(codes, S), synth.FS, 1e5)):
        want = to.filter_data_edge(x, fs, fc, poles)
        got = filters.bessel_filtfilt_odd(torch.from_numpy(x.astype(np.float32)).cuda(), fs, fc, poles).cpu().numpy()
        assert got.shape == x.shape
        assert np.abs(got - want).max() <= max(1e-5 * np.abs(want).max(), 2e-6)


def test_linearity_and_dc_gain():
    # constant input -> constant output (DC gain exactly 1, steady-state boundaries)
    codes = np.full(50000, 40000, np.uint16) & np.uint16(filters.chimera_bitmask(S))
    y = gpu_filter(codes, 1e5, 8)
    assert np.ptp(y) == 0 and np.isclose(y[0], to.scale_raw_data(codes[:1], S)[0], rtol=1e-7)


def test_forward_only_matches_lfilter():
    codes, _ = synth.c1_trace(n=100000, n_events=20, seed=4)
    x = to.scale_raw_data(codes, S)
    b, a = bessel(8, 2 * 1e5 / synth.FS, "low")
    med = np.median(x)
    want, _ = lfilter(b, a, x, zi=lfilter_zi(b, a) * med)
    got = gpu_filter(codes, 1e5, 8, forward_only=True, padding=0)
    check(got, want)


def test_float_input_path():
    codes, _ = synth.c1_trace(n=120000, n_events=25, seed=6)
    x = to.scale_raw_data(codes, S)
    med = float(np.median(x))
    want = to.filter_data(x, synth.FS, 1e5, 8)
    xt = torch.from_numpy(x.astype(np.float32)).cuda()
    got = filters.bessel_filtfilt(xt, synth.FS, 1e5, 8, pad_value=med).cpu().numpy()
    check(got, want)
    # plain zero-state lfilter
    b, a = bessel(8, 2 * 1e5 / synth.FS, "low")
    want2 = lfilter(b, a, x - med)
    got2 = filters.bessel_lfilter(torch.from_numpy((x - med).astype(np.float32)).cuda(), synth.FS, 1e5, 8).cpu().numpy()
    assert np.abs(got2 - want2).max() < ABS_TOL


def test_code_median_is_exact():
    rng = np.random.default_rng(11)
    for n in (1, 2, 1001, 65536, 5_000_001):
        codes = (rng.normal(40000, 60, n).astype(np.int64) & 0xFFFC).astype(np.uint16)
        c1, c2 = median.code_median(torch.from_numpy(codes).cuda(), 0xFFFC)
        srt = np.sort(codes)
        assert (c1, c2) == (int(srt[(n - 1) // 2]), int(srt[n // 2]))
    # bimodal, 1 000 001 codes: under 2^21 samples the stride is 1 and the estimate's full histogram is already exact
    # (the window search over the device counters is test_gpu_median_kernels.py's)
    codes = np.concatenate((np.full(500000, 1000), np.full(500001, 60000))).astype(np.uint16)
    assert median.code_median(torch.from_numpy(codes).cuda(), 0xFFFF) == (60000, 60000)


def test_large_trace_properties():
    """2^27 samples generated on the device: time-reversal symmetry of the zero-phase
    filter (filtfilt(reverse(x)) == reverse(filtfilt(x))) and agreement with the oracle on
    an interior window."""
    n = 1 << 27
    raw = synth.device_trace(n, "cuda", seed=99)
    c1, c2 = median.code_median(raw, filters.chimera_bitmask(S))
    y = filters.dequant_filtfilt(raw, S, 1e5, 8, median_codes=(c1, c2))
    yr = filters.dequant_filtfilt(torch.flip(raw.view(torch.int16), [0]).view(torch.uint16).contiguous(), S, 1e5, 8, median_codes=(c1, c2))
    assert torch.max(torch.abs(torch.flip(yr, [0]) - y)).item() < 0.05
    lo, hi = 50_000_000, 50_300_000
    win = raw[lo - 5000:hi + 5000].cpu().numpy()
    x = to.scale_raw_data(win, S)
    want = to.filter_data(x, synth.FS, 1e5, 8)[5000:-5000]
    got = y[lo:hi].cpu().numpy()
    assert np.abs(got - want).max() < ABS_TOL


def test_integration_stub_binds_the_c_abi_directly():
    """INTEGRATION.md section 2: a maintainer's own ctypes binding of ct_filtfilt_u16 (own CDLL handle, own mirror of
    CtFilterCoef, argtypes as written there) gives the package's result bit for bit."""
    import ctypes as C
    from cusumtools_b200 import _lib

    class Coef(C.Structure):
        _fields_ = [("nsec", C.c_int32), ("order", C.c_int32), ("na1", C.c_float * 5), ("na2", C.c_float * 5),
                    ("ss", C.c_float * 5), ("fir", C.c_float * 11), ("gain", C.c_float)]

    L = C.CDLL(_lib.LIB_PATH)
    L.ct_last_error.restype = C.c_char_p
    assert L.ct_version() == 2
    L.ct_filtfilt_u16.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_float, C.c_uint16, C.c_float, C.c_float,
                                  C.POINTER(Coef), C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    L.ct_filtfilt_workspace_bytes.restype = C.c_int64
    L.ct_filtfilt_workspace_bytes.argtypes = [C.c_int64, C.c_int64, C.c_int]
    S = synth.CHIMERA_SETTINGS
    codes, _ = synth.c1_trace(n=700_001, n_events=100, seed=21)
    raw = torch.from_numpy(codes).cuda()
    want = filters.dequant_filtfilt(raw, S, 1e5, 8)
    design = bessel_lowpass(8, 2 * 1e5 / synth.FS)
    theirs = filters.make_coef(design)
    assert C.sizeof(Coef) == C.sizeof(theirs)
    coef = Coef.from_buffer_copy(bytes(theirs))
    H = filters.warmup_samples(design)
    mask = filters.chimera_bitmask(S)
    alpha, _ = filters.chimera_affine(S)
    c1, c2 = median.code_median(raw, mask)
    median_code = 0.5 * (c1 + c2)
    pad_value = float(np.median(filters.scale_codes_host(np.array([c1, c2], dtype=np.uint16), S)))
    out = torch.empty(raw.numel(), dtype=torch.float32, device="cuda")
    wsb = L.ct_filtfilt_workspace_bytes(raw.numel(), 1000, H)
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    rc = L.ct_filtfilt_u16(raw.data_ptr(), raw.numel(), 1000, median_code, mask, alpha, pad_value, C.byref(coef), H, 0,
                           out.data_ptr(), ws.data_ptr(), wsb, None, torch.cuda.current_stream().cuda_stream)
    assert rc == 0, L.ct_last_error().decode()
    torch.cuda.synchronize()
    assert torch.equal(out, want)
