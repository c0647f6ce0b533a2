"""Exact median of the masked ADC codes: the pad value of the reference's np.pad(mode='median') (plot-trace.py:319).

A strided-sample histogram (summed over the ranks of `group`) gives an estimate; the exact counts of the codes below
and inside an 8-code window at `est - 3 step` pin the two middle order statistics, or say which way the window moves
(6 steps; after the first miss the estimate is made again from all the data).  A distribution no window catches takes
the full histogram.  The counts come from the forward filter pass, from their own kernel or from the host loop
(`route`); with `group=None` nothing is communicated.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import NamedTuple

import numpy as np
import torch

from . import _lib


def _world(group) -> int:
    import torch.distributed as dist
    return dist.get_world_size(group)


def _all_reduce_(t: torch.Tensor, group) -> torch.Tensor:
    if group is not None:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t


def _stream(t: torch.Tensor) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


@dataclass
class MedianPlan:
    """State of the exact-median search between its two phases (estimate, verify)."""
    n: int                      # samples of all ranks
    k1: int                     # ranks of the two middle order statistics
    k2: int
    step: int                   # spacing of the masked codes
    shift: int
    est: int                    # estimated median code (a multiple of step)
    lo: int                     # first code of the 8-code verification window
    exact: tuple[int, int] | None = None     # already exact (small traces: full histogram)
    se: float = float("inf")    # standard error of the estimate in code steps: sqrt(sampled) / (2 x samples at the estimate)


def mask_step(mask: int) -> tuple[int, int]:
    """(shift, step): the spacing of the masked codes, step = 1 << shift."""
    shift = 0
    while shift < 16 and not (mask >> shift) & 1:
        shift += 1
    return shift, 1 << shift


class PlanBuffer:
    """Where the device rank search leaves its CtMedianPlan (`dev`, read by ct_filter_forward_planned_u16) and the pinned
    host copy the host reads it from; reusable from one estimate to the next."""

    def __init__(self, device):
        nbytes = C.sizeof(_lib.CtMedianPlan)
        self.dev = torch.empty(nbytes, dtype=torch.uint8, device=device)
        self.host = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
        self.copied = torch.cuda.Event()


class Estimate:
    """Phase 1 under way.  `plan_dev`: the device CtMedianPlan the stream holds once the rank search has run (None when
    the estimate was made on the host); `result()` waits for its host copy only, so kernels that take `plan_dev` can be
    queued before it."""

    def __init__(self, plan: MedianPlan | None = None, buf: PlanBuffer | None = None, n: int | None = None,
                 shift: int = 0, step: int = 1):
        self._plan, self._buf, self._n, self._shift, self._step = plan, buf, n, shift, step
        self.plan_dev = buf.dev if buf is not None else None

    def result(self) -> MedianPlan:
        if self._plan is None:
            self._buf.copied.synchronize()
            p = _lib.CtMedianPlan.from_buffer_copy(self._buf.host.numpy())
            n = self._n if self._n is not None else int(p.n)
            if n == 0:
                raise ValueError("median of an empty trace")
            self._plan = MedianPlan(n, (n - 1) // 2, n // 2, self._step, self._shift, int(p.est), int(p.lo), se=float(p.se))
        return self._plan


def estimate(n_local: int, mask: int, hist_fn, group=None, n_sampled: int | None = None) -> MedianPlan:
    """Phase 1: a strided-sample histogram (summed over `group`) locates the median code.  `n_sampled`:
    the histogram covers only that many of the rank's samples (streaming: the first chunk), so it
    is an estimate even for small traces."""
    return estimate_start(n_local, mask, hist_fn, group, n_sampled).result()


def estimate_start(n_local: int, mask: int, hist_fn, group=None, n_sampled: int | None = None,
                   buf: PlanBuffer | None = None) -> Estimate:
    """`estimate` without waiting for its result: a device histogram is ranked on the device into `buf` (or a new
    PlanBuffer), which is then copied to the host behind an event."""
    shift, step = mask_step(mask)
    if group is None:
        n = int(n_local)
        if n == 0:
            raise ValueError("median of an empty trace")
        stride = max(1, (n if n_sampled is None else int(n_sampled)) // (1 << 20))  # ~1 M samples: median s.e. < 0.1 code
        hist = hist_fn(stride)
    else:
        # every rank samples with the stride of ITS share (ranks own equal shares), and the sample count rides in the
        # same all_reduce as the histogram: one collective for the phase
        stride = max(1, (int(n_local) if n_sampled is None else int(n_sampled)) * _world(group) // (1 << 20))
        h = hist_fn(stride).to(torch.int64)
        packed = _all_reduce_(torch.cat((h, torch.tensor([int(n_local)], dtype=torch.int64, device=h.device))), group)
        hist, n = packed[:-1], None                        # (the total comes back with the rank search: one read)
    exact = stride == 1 and n_sampled is None
    if group is not None and (exact or not hist.is_cuda):
        n = int(packed[-1].item())
    if exact:
        if n == 0:
            raise ValueError("median of an empty trace")
        k1, k2 = (n - 1) // 2, n // 2
        cdf = torch.cumsum(hist.to(torch.int64), 0)
        want = torch.tensor([k1 + 1, k2 + 1], dtype=torch.int64, device=cdf.device)
        c1, c2 = (int(v) for v in torch.searchsorted(cdf, want).tolist())
        return Estimate(MedianPlan(n, k1, k2, step, shift, c1, max(0, c1 - 3 * step), exact=(c1, c2)))
    # the rank search runs where the histogram lives: a 56-byte CtMedianPlan comes back instead of 65 536 bins (with the
    # total of all ranks in it: one read); ct_median_plan computes est, lo and se as the host branch below does
    if hist.is_cuda and hist.dtype in (torch.int32, torch.int64) and hist.is_contiguous():
        buf = buf if buf is not None else PlanBuffer(hist.device)
        with torch.cuda.device(hist.device):
            rc = _lib.lib().ct_median_plan(hist.data_ptr(), int(hist.dtype == torch.int64), shift,
                                           packed[-1:].data_ptr() if n is None else None, buf.dev.data_ptr(), _stream(hist))
            _lib.check(rc, "ct_median_plan")
            buf.host.copy_(buf.dev, non_blocking=True)
            buf.copied.record()
        return Estimate(buf=buf, n=n, shift=shift, step=step)
    # (CPU tensors: the gloo tests of the host logic)
    hist = hist.to(torch.int64)
    cdf = torch.cumsum(hist, 0)
    idx = torch.searchsorted(cdf, (cdf[-1:] + 1) // 2).clamp_(max=hist.numel() - 1)
    i, dens, total = (int(v) for v in torch.cat((idx, hist[idx], cdf[-1:])).tolist())
    if n == 0:
        raise ValueError("median of an empty trace")
    k1, k2 = (n - 1) // 2, n // 2
    est = (i >> shift) * step
    # the sample median of m samples with density f at the median has s.e. 1 / (2 f sqrt(m)); f = dens / m per code step
    se = 0.5 * float(np.sqrt(max(total, 1))) / max(dens, 1)
    return Estimate(MedianPlan(n, k1, k2, step, shift, est, max(0, est - 3 * step), se=se))


def verify(plan: MedianPlan, counts9, group=None):
    """Phase 2: the exact counts of the codes below / inside the window (summed over `group`) either pin
    the two middle order statistics or say which way the window has to move (returns None, new lo)."""
    c = _all_reduce_(counts9.to(torch.int64), group).cpu().numpy().astype(np.int64)
    below, cw = int(c[0]), int(c[0]) + np.cumsum(c[1:])
    if below <= plan.k1 and plan.k2 < cw[-1]:
        return (plan.lo + int(np.searchsorted(cw, plan.k1 + 1)) * plan.step,
                plan.lo + int(np.searchsorted(cw, plan.k2 + 1)) * plan.step), plan.lo
    return None, (max(0, plan.lo - 6 * plan.step) if plan.k1 < below else plan.lo + 6 * plan.step)


def search(n_local: int, mask: int, hist_fn, count_fn, group=None, plan: MedianPlan | None = None,
           first_counts=None) -> tuple[int, int]:
    """Host side of the exact global median: the two middle order statistics of the masked
    codes of ALL ranks.  `hist_fn(stride)` returns this rank's strided-sample histogram
    (int tensor[65536]) and `count_fn(lo, step)` its 9 window counters (#codes < lo, then
    #codes == lo + i*step); both are summed over `group` here, so every rank takes the same
    decisions and returns the same pair.  (The device kernels are passed in, which is what
    lets the world-size-2 gloo test drive this logic on CPU.)  `plan` / `first_counts`: an
    estimate already made and the window counts a fused kernel already produced for it."""
    if plan is None:
        plan = estimate(n_local, mask, hist_fn, group)
    if plan.exact is not None:
        return plan.exact
    counts = first_counts
    for attempt in range(16):
        if counts is None:
            counts = count_fn(plan.lo, plan.step)
        pair, plan.lo = verify(plan, counts, group)
        if pair is not None:
            return pair
        if attempt == 0:
            # the window missed: the estimate came from too small or too local a sample (streaming: the first
            # piece of a drifting trace).  Re-estimate from a strided histogram of ALL the data before stepping.
            again = estimate(n_local, mask, hist_fn, group)
            if again.exact is not None:
                return again.exact
            plan.lo = again.lo                 # (plan.est stays: the filter has already subtracted it)
        counts = None
    cdf = np.cumsum(_all_reduce_(hist_fn(1).to(torch.int64), group).cpu().numpy())   # pathological distribution
    return int(np.searchsorted(cdf, plan.k1 + 1)), int(np.searchsorted(cdf, plan.k2 + 1))


def count_window(raw: torch.Tensor, mask: int, lo: int, step: int, counts: torch.Tensor, nbins: int = 8) -> torch.Tensor:
    """Add the window counts of the codes in `raw` to `counts` (int64[9] on the device: #codes < lo, then
    #codes == lo + i*step): eight codes, or only the first four with `nbins=4` (counts[5:] untouched)."""
    if raw.numel():
        L = _lib.lib()
        count = L.ct_count_window4_u16 if nbins == 4 else L.ct_count_window_u16
        _lib.check(count(raw.data_ptr(), raw.numel(), mask, lo, step, counts.data_ptr(), _stream(raw)), "ct_count_window_u16")
    return counts


def verify_on_device(plan: MedianPlan, counts: torch.Tensor, nbins: int, result: torch.Tensor, group=None) -> None:
    """Phase 2 without a host round trip: the counts (summed over `group` on the stream) become
    CtMedianResult {code1, code2, pad_x = median - plan.est (float bits), status} in `result` (int32[4]),
    evaluated by one device thread.  status != 0: the window missed the median."""
    _all_reduce_(counts, group)
    rc = _lib.lib().ct_median_verify(counts.data_ptr(), nbins, plan.k1, plan.k2, plan.lo, plan.step, float(plan.est),
                                     result.data_ptr(), _stream(counts))
    _lib.check(rc, "ct_median_verify")


def device_counters(raw: torch.Tensor, mask: int, hist: torch.Tensor | None = None):
    """(hist_fn, count_fn) of `search` over the codes of `raw` (this rank's owned samples).  `hist`: an int32[65536]
    device buffer that hist_fn zeroes and fills (each histogram is consumed on the stream before the next is made)."""
    def hist_fn(stride):
        h = torch.zeros(65536, dtype=torch.int32, device=raw.device) if hist is None else hist.zero_()
        if raw.numel():
            _lib.check(_lib.lib().ct_hist_sampled_u16(raw.data_ptr(), raw.numel(), stride, mask, h.data_ptr(), _stream(raw)),
                       "ct_hist_sampled_u16")
        return h

    def count_fn(lo, step):
        return count_window(raw, mask, lo, step, torch.zeros(9, dtype=torch.int64, device=raw.device))

    return hist_fn, count_fn


class Route(NamedTuple):
    count: str | None    # where the window counts come from: "ride" (the forward pass), "kernel" (count_window), None
    device: bool         # verify_on_device decides (else search, on the host)
    lo: int              # the window: its first code and how many codes it counts
    nbins: int


def route(plan: MedianPlan, *, fixed: bool = False, streamed: bool = False, fused_count: bool = True) -> Route:
    """How the analyzer gets from `plan` to the exact median.  Nothing to count when the plan is already exact or the
    caller has the median (`fixed`).  The estimate of a resident trace comes from a sample of ALL of it, on every rank
    the same, and `plan.se` is its standard error in code steps.  Up to 0.8 the eight-code window est - 3 .. est + 4
    holds the median (4 sigma) and is verified on the device; the count rides on the forward pass (`fused_count`,
    4.1 instructions per code, codes at most 4 apart) or runs as its own kernel (four codes est - 1 .. est + 2 when
    se <= 0.25).  Beyond that - a drifting baseline - or from a partial trace (`streamed`): the host loop, starting from
    an eight-code count of its own kernel."""
    if plan.exact is not None or fixed:
        return Route(None, False, plan.lo, 8)
    if streamed or plan.se > 0.8:
        return Route("kernel", False, plan.lo, 8)
    if fused_count and plan.step <= 4:
        return Route("ride", True, plan.lo, 8)
    if plan.se <= 0.25:
        return Route("kernel", True, max(0, plan.est - plan.step), 4)
    return Route("kernel", True, plan.lo, 8)


def code_median(raw: torch.Tensor, mask: int = 0xFFFF, group=None) -> tuple[int, int]:
    """The two middle order statistics (equal for odd n) of the masked codes, exactly; with `group`, of the
    codes of every rank when each passes the samples it owns.  Synchronises with the host for the rank search and for
    each window count."""
    if raw.dtype not in (torch.uint16, torch.int16):
        raise TypeError("raw must hold the 16-bit ADC codes (torch.uint16 or the int16 view)")
    if not raw.is_cuda:
        raise RuntimeError("raw must be a CUDA tensor: cusumtools_b200 has no CPU path")
    if not raw.is_contiguous():
        raise ValueError("raw must be contiguous")
    return search(raw.numel(), mask, *device_counters(raw, mask), group)
