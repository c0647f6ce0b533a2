"""Stage 3b of the hot path: batched step-response fit of short events (GPU), rate.csv / events.csv type 1.

The reference has no implementation (readevents.py:1334-1337 reads a type-1 event file with the columns time,
current, cusum, stepfit; events.csv carries `rc_const1_us` / `rc_const2_us`); definition of record:
oracle/stepfit_oracle.py.  For window sample t and p = (i0, a, u1, u2, tau1, tau2):

    f(t) = i0 - a (1 - exp(-(t-u1)/tau1)) H(t-u1) + a (1 - exp(-(t-u2)/tau2)) H(t-u2),   H(s) = [s >= 0]

fitted by Levenberg-Marquardt, one warp per event (ct_stepfit_batch).  Events shorter than a few rise times of the
zero-phase filter have no plateau CUSUM+ could measure; the fit recovers their depth from the edges."""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from .cusum import LevelTable
from .design import bessel_lowpass
from .filters import _require_cuda, _stream_ptr

TYPE_STEPFIT, TYPE_STEPFIT_FAILED = 1, 7
DEFAULT_MAX_ITERS = 50
MAX_WINDOW = _lib.STEPFIT_MAX_WINDOW


@dataclass
class StepFitTable:
    """Per-event fit.  params[e] = (i0 pA, a pA, u1, u2, tau1, tau2 samples, relative to the window start); cost = sum
    of squared residuals (pA^2) at the fit; iters = LM trials (the initial evaluation and every trial, evaluated or
    not: a trial without a positive-definite matrix or outside the domain still counts); status = 1 (valid fit), 7 (fit failed), or the
    event's type if it was not fitted (its row is then zero)."""
    params: torch.Tensor       # float64 [E, 6]
    cost: torch.Tensor         # float64 [E]
    iters: torch.Tensor        # int32 [E]
    status: torch.Tensor       # int32 [E]
    levels: LevelTable | None = None     # the three level rows of every valid fit (standalone calls)


def zero_phase_rise_tau(samplerate: float, cutoff: float, order: int = 8) -> float:
    """tau0 of the initial guess: (t90 - t10) / ln 9 in samples, t10 / t90 the first samples at which the step
    response of the zero-phase filter (forward and backward Bessel pass), computed in float64 from the design,
    reaches 10 % / 90 %.  38 samples, tau0 = 17.3, at 100 kHz / 8 poles / 4.17 MHz."""
    d = bessel_lowpass(int(order), 2.0 * float(cutoff) / float(samplerate))
    h = d._impulse(max(256, d.impulse_tail(1e-12)))
    g = np.convolve(h, h[::-1])                  # impulse response of filtfilt, centred at len(h) - 1
    s = np.cumsum(g)
    s /= s[-1]
    t10, t90 = int(np.argmax(s >= 0.1)), int(np.argmax(s >= 0.9))
    return float((t90 - t10) / math.log(9.0))


def select_short(win_start: torch.Tensor, win_end: torch.Tensor, types: torch.Tensor, *, padding: int,
                 stepfit_samples: int, n_events_dev: torch.Tensor | None = None) -> None:
    """In place: accepted events (type 0) with end - start < stepfit_samples become type 1 (ct_stepfit_select)."""
    _require_cuda(types, "types", torch.int32)
    with torch.cuda.device(types.device):
        rc = _lib.lib().ct_stepfit_select(win_start.data_ptr(), win_end.data_ptr(), types.data_ptr(),
                                          n_events_dev.data_ptr() if n_events_dev is not None else None, types.numel(),
                                          int(padding), int(stepfit_samples), _stream_ptr(types))
    _lib.check(rc, "ct_stepfit_select")


def launch(y: torch.Tensor, win_start: torch.Tensor, win_end: torch.Tensor, types: torch.Tensor, out: dict, levels: dict, *,
           padding: int, tau0: float, max_iters: int = DEFAULT_MAX_ITERS, n_events_dev: torch.Tensor | None = None,
           capacity: int | None = None) -> None:
    """ct_stepfit_batch into caller-owned buffers: out = {params, cost, iters}, levels = {n_levels, edges, mean, std}
    (`max_levels` = mean.shape[1]).  `types` is updated in place (7 where a fit fails)."""
    cap = int(types.numel() if capacity is None else capacity)
    with torch.cuda.device(y.device):
        rc = _lib.lib().ct_stepfit_batch(
            y.data_ptr(), y.numel(), win_start.data_ptr(), win_end.data_ptr(), types.data_ptr(),
            n_events_dev.data_ptr() if n_events_dev is not None else None, cap, int(padding), float(tau0), int(max_iters),
            int(levels["mean"].shape[1]), out["params"].data_ptr(), out["cost"].data_ptr(), out["iters"].data_ptr(),
            levels["n_levels"].data_ptr(), levels["edges"].data_ptr(), levels["mean"].data_ptr(), levels["std"].data_ptr(),
            _stream_ptr(y))
    _lib.check(rc, "ct_stepfit_batch")


def step_fit(y: torch.Tensor, win_start: torch.Tensor, win_end: torch.Tensor, *, padding: int, tau0: float,
             max_iters: int = DEFAULT_MAX_ITERS, types: torch.Tensor | None = None, max_levels: int = 3) -> StepFitTable:
    """Step-response fit of every event window y[win_start[e]:win_end[e]) (device int64 index tensors) whose `types`
    entry is 1 (all of them when `types` is None), one warp per event.  `padding` baseline samples lead and trail
    the event in each window; `tau0` (samples) starts both rise times (`zero_phase_rise_tau`)."""
    _require_cuda(y, "y", torch.float32)
    _require_cuda(win_start, "win_start", torch.int64)
    _require_cuda(win_end, "win_end", torch.int64)
    E = win_start.numel()
    if win_end.numel() != E:
        raise ValueError("win_start and win_end differ in length")
    dev = y.device
    if types is None:
        st = torch.full((E,), TYPE_STEPFIT, dtype=torch.int32, device=dev)
    else:
        _require_cuda(types, "types", torch.int32)
        st = types.clone()
    out = {"params": torch.zeros((E, 6), dtype=torch.float64, device=dev),
           "cost": torch.zeros(E, dtype=torch.float64, device=dev),
           "iters": torch.zeros(E, dtype=torch.int32, device=dev)}
    lv = {"n_levels": torch.zeros(E, dtype=torch.int32, device=dev),
          "edges": torch.full((E, max_levels + 1), -1, dtype=torch.int32, device=dev),
          "mean": torch.zeros((E, max_levels), dtype=torch.float64, device=dev),
          "std": torch.zeros((E, max_levels), dtype=torch.float64, device=dev)}
    if E:
        launch(y, win_start, win_end, st, out, lv, padding=padding, tau0=tau0, max_iters=max_iters)
    levels = LevelTable(lv["n_levels"], lv["edges"], lv["mean"], lv["std"], torch.zeros(E, dtype=torch.uint8, device=dev),
                        int(max_levels))
    return StepFitTable(out["params"], out["cost"], out["iters"], st, levels)


def stepfit_flat(samples: torch.Tensor, offsets: torch.Tensor, **kw) -> StepFitTable:
    """Pre-extracted events in one flat buffer: event e is samples[offsets[e]:offsets[e+1]], each with `padding`
    baseline samples on both sides."""
    _require_cuda(offsets, "offsets", torch.int64)
    return step_fit(samples, offsets[:-1].contiguous(), offsets[1:].contiguous(), **kw)


def rc_constants_us(params: np.ndarray, samplerate: float) -> tuple[np.ndarray, np.ndarray]:
    """events.csv rc_const1_us / rc_const2_us from the fitted rise times (samples)."""
    p = np.asarray(params, np.float64).reshape(-1, 6)
    return p[:, 4] * (1e6 / float(samplerate)), p[:, 5] * (1e6 / float(samplerate))


def model(params, n: int) -> np.ndarray:
    """f(t), t = 0 .. n-1, of one parameter row (float64; the `stepfit` column of a type-1 event file)."""
    i0, a, u1, u2, t1, t2 = (float(v) for v in params)
    t = np.arange(int(n), dtype=np.float64)
    s1, s2 = t - u1, t - u2
    with np.errstate(over="ignore"):
        q1 = np.where(s1 >= 0, -np.expm1(-np.maximum(s1, 0.0) / t1), 0.0)
        q2 = np.where(s2 >= 0, -np.expm1(-np.maximum(s2, 0.0) / t2), 0.0)
    return i0 - a * q1 + a * q2
