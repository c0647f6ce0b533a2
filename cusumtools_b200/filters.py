"""Stage 1 of the hot path: dequantise + median pad + zero-phase Bessel low-pass.

Python entry points over the C ABI (include/cusumtools_b200.h).  They mirror the
reference call sites `App.scale_raw_data` / `App.filter_data`
(plot-trace.py:272-287, 313-320) and `scipy.signal.lfilter`/`filtfilt` as used there;
torch is used only for device memory and streams.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

from . import _lib, median
from .design import BesselDesign, bessel_lowpass

DEFAULT_HALO_EPS = 1e-7      # truncated natural response relative to max |x - median|


# ------------------------------------------------------------------ coefficient packing
_coef_cache: dict[tuple[int, float], "_lib.CtFilterCoef"] = {}


def make_coef(design: BesselDesign) -> _lib.CtFilterCoef:
    """Pack a design for the kernel: per-section taps, steady-state factors, gain."""
    key = (design.order, design.wn)
    if key not in _coef_cache:
        _coef_cache[key] = _make_coef(design)
    return _coef_cache[key]


def _make_coef(design: BesselDesign) -> _lib.CtFilterCoef:
    """H(z) = gain (1 + z^-1)^order / prod (1 - na1 z^-1 - na2 z^-2): the kernel runs the all-pole sections at every
    sample and the numerator as ONE binomial FIR (with the gain folded in) only where it is needed.  The gain is
    evaluated from the float32-rounded denominators, so the float32 cascade's DC gain is exactly 1."""
    k = _lib.CtFilterCoef()
    k.nsec = design.nsec
    order = 0
    inv = 1.0           # DC gain of the all-pole sections up to and including the current one
    for s in range(design.nsec):
        a1, a2 = design.sections[s]
        k.na1[s], k.na2[s] = -a1, -a2
        den = 1.0 - float(k.na1[s]) - float(k.na2[s])          # from the values the kernel will use
        inv /= den
        k.ss[s] = inv
        order += 1 if bool(design.first_order[s]) else 2
    k.order = order
    gain = 1.0 / (inv * 2.0 ** order)
    k.gain = gain
    for i in range(order + 1):
        k.fir[i] = gain * math.comb(order, i)
    peak = 65536.0 * inv  # largest un-normalised intermediate for a full-scale step
    if not math.isfinite(peak) or peak > 1e36:
        raise ValueError("cutoff/samplerate too low for the float32 cascade (intermediate overflow)")
    return k


def warmup_samples(design: BesselDesign, eps: float = DEFAULT_HALO_EPS) -> int:
    """IIR warm-up H of a run: the cascade's impulse response is below eps beyond it."""
    return max(1, design.impulse_tail(eps))


def scratch_decimation(design: BesselDesign, padding: int = 1000, eps: float = DEFAULT_HALO_EPS) -> int:
    """Every how-many-th forward sample the scratch between the two passes keeps (1, 2 or 4): the library's
    choice from the cascade's stop band (aliasing error < 1e-7), reported for diagnostics and benchmarks."""
    return int(_lib.lib().ct_filter_decimation(C.byref(make_coef(design)), int(padding), warmup_samples(design, eps)))


def _workspace(n: int, padding: int, H: int, forward_only: bool, device, workspace):
    """Device scratch for the forward output (caller may pass a reusable uint8 tensor)."""
    if forward_only:
        return None, 0
    need = int(_lib.lib().ct_filtfilt_workspace_bytes(n, padding, H))
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty(need, dtype=torch.uint8, device=device)
    return workspace, need


def _stream_ptr(t: torch.Tensor) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _require_cuda(t: torch.Tensor, name: str, dtype) -> None:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: cusumtools_b200 has no CPU path")
    if t.dtype != dtype:
        raise TypeError(f"{name} must have dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")


# ------------------------------------------------------------------- Chimera scaling
def chimera_bitmask(settings) -> int:
    """plot-trace.py:281: bitmask = (2**16 - 1) - (2**(16-ADCbits) - 1)."""
    bits = int(np.squeeze(settings["SETUP_ADCBITS"]))
    return (2 ** 16 - 1) - (2 ** (16 - bits) - 1)


def scale_codes_host(codes, settings) -> np.ndarray:
    """The reference's own operation sequence (plot-trace.py:280-287) applied on the host
    to a handful of codes: used for the pad value so it is bit-identical to
    np.median(scale_raw_data(raw))."""
    TIAgain = np.squeeze(settings["SETUP_TIAgain"])
    preADCgain = np.squeeze(settings["SETUP_preADCgain"])
    currentoffset = np.squeeze(settings["SETUP_pAoffset"])
    ADCvref = np.squeeze(settings["SETUP_ADCVREF"])
    closedloop_gain = TIAgain * preADCgain
    t = np.asarray(codes).astype(np.uint16) & chimera_bitmask(settings)
    t = ADCvref - (2 * ADCvref) * t.astype(float) / float(2 ** 16)
    t = -t / float(closedloop_gain) + float(currentoffset)
    return t * 1e12


def chimera_affine(settings) -> tuple[float, float]:
    """pA = alpha * (code & mask) + beta, the closed form of plot-trace.py:283-287."""
    b0, b1 = scale_codes_host(np.array([0, 32768], dtype=np.uint16), settings)
    return float((b1 - b0) / 32768.0), float(b0)


# ------------------------------------------------------------------------ entry points
def filtfilt_codes(raw: torch.Tensor, *, alpha: float, pad_value: float, median_code: float, mask: int,
                   design: BesselDesign, padding: int = 1000, forward_only: bool = False,
                   halo_eps: float = DEFAULT_HALO_EPS,
                   out: torch.Tensor | None = None, workspace: torch.Tensor | None = None, stats=None) -> torch.Tensor:
    """out = pad_value + alpha * filtfilt((raw & mask) - median_code) with the reference's
    boundary handling (dequantisation fused into the load and the store).  `stats`: a
    `_lib.CtFilterStats` to have the baseline block sums of the output tallied on the way
    out (detect.Baseline.stats_args; needs block % stats_granule == 0)."""
    if raw.dtype not in (torch.uint16, torch.int16):
        raise TypeError("raw must hold the 16-bit ADC codes (torch.uint16 or the int16 view)")
    _require_cuda(raw, "raw", raw.dtype)
    n = raw.numel()
    if out is None:
        out = torch.empty(n, dtype=torch.float32, device=raw.device)
    _require_cuda(out, "out", torch.float32)
    if out.numel() != n:
        raise ValueError("out has the wrong length")
    coef = make_coef(design)
    H = warmup_samples(design, halo_eps)
    ws, wsb = _workspace(n, int(padding), H, forward_only, raw.device, workspace)
    with torch.cuda.device(raw.device):
        rc = _lib.lib().ct_filtfilt_u16(raw.data_ptr(), n, int(padding), float(median_code), int(mask),
                                        float(alpha), float(pad_value), C.byref(coef), H,
                                        int(bool(forward_only)), out.data_ptr(), ws.data_ptr() if ws is not None else None,
                                        wsb, C.byref(stats) if stats is not None else None, _stream_ptr(raw))
    _lib.check(rc, "ct_filtfilt_u16")
    return out


def dequant_filtfilt(raw: torch.Tensor, settings, cutoff: float, order: int = 8, *,
                     samplerate: float | None = None, padding: int = 1000, forward_only: bool = False,
                     halo_eps: float = DEFAULT_HALO_EPS,
                     median_codes: tuple[int, int] | None = None,
                     out: torch.Tensor | None = None, workspace: torch.Tensor | None = None, stats=None) -> torch.Tensor:
    """`App.scale_raw_data` + `App.filter_data` (plot-trace.py:272-287, 313-320) fused:
    raw Chimera codes on the GPU -> filtered pA (float32) on the GPU.

    `settings` is the dict `scipy.io.loadmat` returns for the `.mat` next to the `.log`
    (or any mapping with the same keys).  `median_codes` lets a multi-GPU caller pass the
    globally reduced median instead of this shard's."""
    fs = float(np.floor(np.squeeze(settings["ADCSAMPLERATE"]))) if samplerate is None else float(samplerate)
    design = bessel_lowpass(int(order), 2.0 * float(cutoff) / fs)
    mask = chimera_bitmask(settings)
    alpha, _ = chimera_affine(settings)
    c1, c2 = median_codes if median_codes is not None else median.code_median(raw, mask)
    vals = scale_codes_host(np.array([c1, c2], dtype=np.uint16), settings)
    pad_value = float(np.median(vals))
    return filtfilt_codes(raw, alpha=alpha, pad_value=pad_value, median_code=0.5 * (c1 + c2), mask=mask,
                          design=design, padding=padding, forward_only=forward_only, halo_eps=halo_eps,
                          out=out, workspace=workspace, stats=stats)


def stats_granule(n: int, padding: int, design: BesselDesign, halo_eps: float = DEFAULT_HALO_EPS) -> int:
    """Baseline blocks must be a multiple of this many samples for the statistics to be fused
    into the filter (one warp group of the lane-sequential passes)."""
    return int(_lib.lib().ct_filtfilt_stats_granule(int(n), int(padding), max(1, design.impulse_tail(halo_eps))))


def float_median(x: torch.Tensor, *, use_abs: bool = False) -> float:
    """Exact np.median of a float32 device vector (float64 mean of the two middle values
    for even n) by a 4-pass most-significant-digit radix select on the GPU."""
    _require_cuda(x, "x", torch.float32)
    n = x.numel()
    if n == 0:
        raise ValueError("median of an empty trace")
    L = _lib.lib()
    st = _stream_ptr(x)

    def select(rank: int) -> float:
        prefix, bits = 0, 0
        for _ in range(4):
            h = torch.zeros(256, dtype=torch.int64, device=x.device)
            _lib.check(L.ct_radix_hist_f32(x.data_ptr(), n, prefix, bits, int(use_abs), h.data_ptr(), st), "ct_radix_hist_f32")
            c = np.cumsum(h.cpu().numpy())
            d = int(np.searchsorted(c, rank + 1))
            rank -= int(c[d - 1]) if d else 0
            prefix, bits = (prefix << 8) | d, bits + 8
        key = np.uint32(prefix)
        b = key ^ (np.uint32(0x80000000) if key & np.uint32(0x80000000) else np.uint32(0xFFFFFFFF))
        return float(np.array([b], dtype=np.uint32).view(np.float32)[0])

    lo = select((n - 1) // 2)
    hi = lo if n % 2 else select(n // 2)
    return float(np.mean(np.array([lo, hi], dtype=np.float64)))


def bessel_filtfilt(x: torch.Tensor, samplerate: float, cutoff: float, order: int = 8, *,
                    pad_value: float | None = None, padding: int = 1000, forward_only: bool = False,
                    halo_eps: float = DEFAULT_HALO_EPS,
                    out: torch.Tensor | None = None, workspace: torch.Tensor | None = None) -> torch.Tensor:
    """Zero-phase Bessel of an already-dequantised float32 trace (e.g. `.bin` data,
    print_trace.py:33): out = pad_value + filtfilt(x - pad_value) with `padding` samples
    of constant pad, i.e. filtfilt(b, a, np.pad(x, padding, constant=pad_value),
    padtype=None)[padding:-padding]; pad_value=None takes the median (the reference's
    `filter_data` on float data)."""
    _require_cuda(x, "x", torch.float32)
    n = x.numel()
    if out is None:
        out = torch.empty(n, dtype=torch.float32, device=x.device)
    _require_cuda(out, "out", torch.float32)
    if out.numel() != n:
        raise ValueError("out has the wrong length")
    if pad_value is None:            # np.pad(mode='median'), plot-trace.py:319
        pad_value = float_median(x)
    design = bessel_lowpass(int(order), 2.0 * float(cutoff) / float(samplerate))
    coef = make_coef(design)
    H = warmup_samples(design, halo_eps)
    ws, wsb = _workspace(n, int(padding), H, forward_only, x.device, workspace)
    with torch.cuda.device(x.device):
        rc = _lib.lib().ct_filtfilt_f32(x.data_ptr(), n, int(padding), float(pad_value), C.byref(coef), H,
                                        int(bool(forward_only)), out.data_ptr(), ws.data_ptr() if ws is not None else None,
                                        wsb, None, _stream_ptr(x))
    _lib.check(rc, "ct_filtfilt_f32")
    return out


def bessel_lfilter(x: torch.Tensor, samplerate: float, cutoff: float, order: int = 8, *,
                   initial: float = 0.0, **kw) -> torch.Tensor:
    """Causal pass only: scipy.signal.lfilter(b, a, x, zi=lfilter_zi(b, a)*initial)[0]
    (`initial = 0` is the plain zero-state lfilter)."""
    return bessel_filtfilt(x, samplerate, cutoff, order, pad_value=float(initial), padding=0,
                           forward_only=True, **kw)


def bessel_filtfilt_odd(x: torch.Tensor, samplerate: float, cutoff: float, poles: int) -> torch.Tensor:
    """legacy/bessel-filter.py:124-131: `np.pad(x, poles, mode='edge')`, scipy's default filtfilt
    (`method='pad', padlen=None`: padtype='odd', padlen = 3*ntaps = 3*(poles+1)) and `[poles:-poles]`,
    so the result has the length of `x`.  The odd extension is a few dozen samples and is built on the
    device with torch; the kernel then runs without a constant pad (which also keeps the scratch at full
    rate), its steady-state initial conditions being exactly scipy's zi*ext[0] and zi*y[-1]."""
    _require_cuda(x, "x", torch.float32)
    p = int(poles)
    xe = torch.cat((x[:1].expand(p), x, x[-1:].expand(p)))
    edge = 3 * (p + 1)
    if xe.numel() <= edge:
        raise ValueError("The length of the input vector x must be greater than padlen")
    left = 2 * xe[0] - torch.flip(xe[1:edge + 1], [0])
    right = 2 * xe[-1] - torch.flip(xe[-edge - 1:-1], [0])
    ext = torch.cat((left, xe, right)).contiguous()
    y = bessel_filtfilt(ext, samplerate, cutoff, p, pad_value=float(ext[0].item()), padding=0)
    return y[edge + p:y.numel() - edge - p]
