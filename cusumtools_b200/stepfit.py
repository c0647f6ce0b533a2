"""Stage 3b of the hot path: batched step-response fit of short events (GPU), rate.csv / events.csv type 1.

The reference has no implementation (readevents.py:1334-1337 reads a type-1 event file with the columns time,
current, cusum, stepfit; events.csv carries `rc_const1_us` / `rc_const2_us`); definition of record:
oracle/stepfit_oracle.py.  For window sample t and p = (i0, a, u1, u2, tau1, tau2):

    f(t) = i0 - a (1 - exp(-(t-u1)/tau1)) H(t-u1) + a (1 - exp(-(t-u2)/tau2)) H(t-u2),   H(s) = [s >= 0]

fitted by Levenberg-Marquardt.  Events shorter than a few rise times of the zero-phase filter have no plateau CUSUM+
could measure; the fit recovers their depth from the edges.  Two kernels run the same fit (the same initial guess, LM
loop, stop tests, validity rule and level rows; oracle/stepfit_twin.py restates it):

* ct_stepfit_batch: one warp per window of at most MAX_WINDOW (8192) samples; `select_short` marks the short events
  (type 1) before CUSUM+, `launch` / `step_fit` fit them;
* ct_stepfit_long_batch: one CTA per window of up to LONG_MAX_WINDOW (131072) samples; `launch_long` / `step_fit_long`.

The fallback (`TraceAnalyzer(stepfit_fallback=True)`) fits the events CUSUM+ leaves without a sub-level, which would
otherwise be type 5: `select_fallback` runs after CUSUM+ and marks them type 1 (window <= MAX_WINDOW) or
TYPE_STEPFIT_LONG (longer), then `launch` and `launch_long` fit them, in that order; a failed fit is type 7."""
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
TYPE_STEPFIT_LONG = _lib.TYPE_STEPFIT_LONG       # long fit pending: internal to the analyzer's step
DEFAULT_MAX_ITERS = 50
# LM trials of the long fit: on long shallow windows the trials accepted and rejected at the kink in u alternate for
# longer, and 50 trials leave about one -180 pA event of 9 000 - 90 000 samples in ten unconverged (type 7)
LONG_DEFAULT_MAX_ITERS = 200
MAX_WINDOW = _lib.STEPFIT_MAX_WINDOW
LONG_MAX_WINDOW = _lib.STEPFIT_LONG_MAX_WINDOW


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

    def rows(self, n: int) -> StepFitTable:
        """The first `n` rows, as views of these buffers."""
        return StepFitTable(self.params[:n], self.cost[:n], self.iters[:n], self.status[:n],
                            None if self.levels is None else self.levels.rows(n))


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


def select_fallback(levels: LevelTable, win_start: torch.Tensor, win_end: torch.Tensor, types: torch.Tensor, *,
                    n_events_dev: torch.Tensor | None = None, capacity: int | None = None) -> None:
    """In place, after CUSUM+: every event still of type 0 with no level overflow and fewer than three levels
    (`levels.n_levels`, `levels.overflow`) becomes type 1 if its window is at most MAX_WINDOW samples, else
    TYPE_STEPFIT_LONG (ct_stepfit_fallback_select).  No other row changes."""
    _require_cuda(types, "types", torch.int32)
    cap = int(types.numel() if capacity is None else capacity)
    with torch.cuda.device(types.device):
        rc = _lib.lib().ct_stepfit_fallback_select(levels.n_levels.data_ptr(), levels.overflow.data_ptr(),
                                                   win_start.data_ptr(), win_end.data_ptr(), types.data_ptr(),
                                                   n_events_dev.data_ptr() if n_events_dev is not None else None, cap,
                                                   _stream_ptr(types))
    _lib.check(rc, "ct_stepfit_fallback_select")


def _launch(fn: str, y, win_start, win_end, types, out, levels, padding, tau0, max_iters, n_events_dev, capacity,
            *extra) -> None:
    cap = int(types.numel() if capacity is None else capacity)
    with torch.cuda.device(y.device):
        rc = getattr(_lib.lib(), fn)(
            y.data_ptr(), y.numel(), win_start.data_ptr(), win_end.data_ptr(), types.data_ptr(),
            n_events_dev.data_ptr() if n_events_dev is not None else None, cap, int(padding), float(tau0), int(max_iters),
            levels.max_levels, out.params.data_ptr(), out.cost.data_ptr(), out.iters.data_ptr(),
            levels.n_levels.data_ptr(), levels.edges.data_ptr(), levels.mean.data_ptr(), levels.std.data_ptr(),
            *extra, _stream_ptr(y))
    _lib.check(rc, fn)


def launch(y: torch.Tensor, win_start: torch.Tensor, win_end: torch.Tensor, types: torch.Tensor, out: StepFitTable,
           levels: LevelTable, *, padding: int, tau0: float, max_iters: int = DEFAULT_MAX_ITERS,
           n_events_dev: torch.Tensor | None = None, capacity: int | None = None) -> None:
    """ct_stepfit_batch into caller-owned buffers: the params, cost and iters of `out` and the n_levels, edges, mean
    and std rows of `levels` (overflow is not touched).  `types` is updated in place (7 where a fit fails)."""
    _launch("ct_stepfit_batch", y, win_start, win_end, types, out, levels, padding, tau0, max_iters, n_events_dev, capacity)


def launch_long(y: torch.Tensor, win_start: torch.Tensor, win_end: torch.Tensor, types: torch.Tensor, out: StepFitTable,
                levels: LevelTable, *, padding: int, tau0: float, max_iters: int = LONG_DEFAULT_MAX_ITERS,
                n_events_dev: torch.Tensor | None = None, capacity: int | None = None,
                row_counter: torch.Tensor | None = None) -> None:
    """ct_stepfit_long_batch, the mirror of `launch`: fits the rows of type TYPE_STEPFIT_LONG (one CTA per event) and
    sets each of them to 1 or 7; rows of every other type are left as they are.  Run it after `launch`.
    `row_counter`: one int64 of device scratch the CTAs claim rows from (allocated here when None)."""
    if row_counter is None:
        row_counter = torch.empty(1, dtype=torch.int64, device=y.device)
    _require_cuda(row_counter, "row_counter", torch.int64)
    _launch("ct_stepfit_long_batch", y, win_start, win_end, types, out, levels, padding, tau0, max_iters, n_events_dev,
            capacity, row_counter.data_ptr())


def _fit_all(fn, selected: int, y, win_start, win_end, padding, tau0, max_iters, types, max_levels) -> StepFitTable:
    _require_cuda(y, "y", torch.float32)
    _require_cuda(win_start, "win_start", torch.int64)
    _require_cuda(win_end, "win_end", torch.int64)
    E = win_start.numel()
    if win_end.numel() != E:
        raise ValueError("win_start and win_end differ in length")
    dev = y.device
    if types is None:
        st = torch.full((E,), selected, dtype=torch.int32, device=dev)
    else:
        _require_cuda(types, "types", torch.int32)
        st = types.clone()
    out = StepFitTable(torch.zeros((E, 6), dtype=torch.float64, device=dev), torch.zeros(E, dtype=torch.float64, device=dev),
                       torch.zeros(E, dtype=torch.int32, device=dev), st, LevelTable.empty(E, max_levels, dev))
    out.levels.clear()
    for t in (out.levels.mean, out.levels.std):
        t.zero_()
    if E:
        fn(y, win_start, win_end, st, out, out.levels, padding=padding, tau0=tau0, max_iters=max_iters)
    return out


def step_fit(y: torch.Tensor, win_start: torch.Tensor, win_end: torch.Tensor, *, padding: int, tau0: float,
             max_iters: int = DEFAULT_MAX_ITERS, types: torch.Tensor | None = None, max_levels: int = 3) -> StepFitTable:
    """Step-response fit of every event window y[win_start[e]:win_end[e]) (device int64 index tensors) whose `types`
    entry is 1 (all of them when `types` is None), one warp per event.  `padding` baseline samples lead and trail
    the event in each window; `tau0` (samples) starts both rise times (`zero_phase_rise_tau`)."""
    return _fit_all(launch, TYPE_STEPFIT, y, win_start, win_end, padding, tau0, max_iters, types, max_levels)


def step_fit_long(y: torch.Tensor, win_start: torch.Tensor, win_end: torch.Tensor, *, padding: int, tau0: float,
                  max_iters: int = LONG_DEFAULT_MAX_ITERS, types: torch.Tensor | None = None,
                  max_levels: int = 3) -> StepFitTable:
    """`step_fit` through the long kernel (one CTA per event, windows up to LONG_MAX_WINDOW samples): every window whose
    `types` entry is TYPE_STEPFIT_LONG (all of them when `types` is None).  Rows of other types keep their type and
    zero rows; a fitted row's status is 1 or 7."""
    return _fit_all(launch_long, TYPE_STEPFIT_LONG, y, win_start, win_end, padding, tau0, max_iters, types, max_levels)


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
