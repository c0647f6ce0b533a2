"""The raw-trace hot path end to end on one GPU or time-sharded over several.

    raw Chimera codes -> [exact global median] -> fused dequantise + Bessel filtfilt
                      -> baseline blocks -> threshold/hysteresis events

One process per GPU.  A rank owns the samples [lo, hi) of the global trace and is handed
them together with `halo` extra samples on each side (read from the shared file / host
buffer, not exchanged: SURVEY.md section 8e).  The only collectives are
  * all_reduce(SUM) of the sampled code histogram and of the 9 window counters that give
    the GLOBAL median pad value (median.py: every rank subtracts the same constant), and
  * all_gather of per-rank event counts (global event ids); event rows stay rank-local.
With `group=None` nothing is communicated and the functions are the single-GPU path.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib, cusum, detect, filters, median, stepfit
from .design import bessel_lowpass
from .median import _all_reduce_


@dataclass
class TraceResult:
    filtered: torch.Tensor          # float32 device, the rank's owned samples only
    baseline: detect.Baseline
    events: detect.EventList        # indices relative to the rank's first owned sample
    pad_value: float
    median_codes: tuple[int, int]
    first_event_id: int = 0         # global id of this rank's first event
    total_events: int = 0


def event_id_offsets(n_local_events: int, group=None, device=None) -> tuple[int, int]:
    """(global id of this rank's first event, total events): ranks own consecutive time
    shards, so ids follow rank order."""
    if group is None:
        return 0, int(n_local_events)
    import torch.distributed as dist
    ws, rk = dist.get_world_size(group), dist.get_rank(group)
    counts = torch.zeros(ws, dtype=torch.int64, device=device)
    counts[rk] = int(n_local_events)
    c = _all_reduce_(counts, group).cpu().numpy()
    return int(c[:rk].sum()), int(c.sum())


def event_ids_and_status(n_local_events: int, status: int, group=None, device=None) -> tuple[int, int, int]:
    """`event_id_offsets` with a status flag riding in the same all_reduce: (first id, total events, sum of the
    ranks' flags).  A rank that hit an error passes status != 0 INSTEAD of raising before the collective, so that
    every rank takes the same decision afterwards (raise together, fall back together) and nobody is left waiting
    in a collective its peers never enter."""
    if group is None:
        return 0, int(n_local_events), int(status)
    import torch.distributed as dist
    ws, rk = dist.get_world_size(group), dist.get_rank(group)
    v = torch.zeros(ws + 1, dtype=torch.int64, device=device)
    v[rk] = int(n_local_events)
    v[ws] = int(status != 0)
    c = _all_reduce_(v, group).cpu().numpy()
    return int(c[:rk].sum()), int(c[:ws].sum()), int(c[ws])


def required_halo(cutoff: float, order: int, samplerate: float, max_event: int, padding: int = 1000,
                  eps: float = filters.DEFAULT_HALO_EPS, block: int = 1) -> int:
    """Samples a rank must read beyond each end of its owned range: IIR warm-up on both
    sides (forward and backward pass) plus one maximal event so that an event straddling
    a shard boundary is seen whole by the rank that owns its start, rounded up to a multiple
    of the baseline `block` (the left halo keeps every rank on the global block grid)."""
    d = bessel_lowpass(int(order), 2.0 * float(cutoff) / float(samplerate))
    h = 2 * max(1, d.impulse_tail(eps)) + int(max_event)
    return -(-h // int(block)) * int(block)


@dataclass
class AnalysisResult:
    """Everything one pass of the hot path over a (shard of a) trace produces; all tensors
    are device-resident views into the analyzer's buffers (valid until its next run)."""
    filtered: torch.Tensor          # float32, the rank's owned samples
    detect_trace: torch.Tensor      # float32, [left halo | owned | right halo]: what the windows refer to
    lo_halo: int                    # samples of detect_trace before the first owned one
    baseline: detect.Baseline
    events: detect.EventList        # indices relative to the rank's first owned sample
    win_start: torch.Tensor         # int64 [E]  CUSUM+ windows [start - padding, end + padding) in detect_trace
    win_end: torch.Tensor           # int64 [E]
    types: torch.Tensor             # int32 [E]  rate.csv type code (0 accepted, >1 rejected)
    levels: "cusum.LevelTable | None"
    pad_value: float
    median_codes: tuple[int, int]
    first_event_id: int = 0
    total_events: int = 0
    intra: "tuple[torch.Tensor, torch.Tensor] | None" = None     # (count int32 [E], pairs int32 [E, 2K]) crossings
    stepfit: "stepfit.StepFitTable | None" = None                # step-response fit of the short events (type 1 / 7)

    def columns(self, index_offset: int = 0) -> dict:
        """The per-event columns by name, in the order of the host event tables (`TraceAnalyzer.tables_to_host`,
        `StreamResult.tables`); `index_offset` is added to starts and ends."""
        starts, ends = self.events.starts, self.events.ends
        if index_offset:
            starts, ends = starts + index_offset, ends + index_offset
        cols = {"starts": starts, "ends": ends, "types": self.types}
        if self.levels is not None:
            lv = self.levels
            cols.update(n_levels=lv.n_levels, edges=lv.edges, mean=lv.mean, std=lv.std, overflow=lv.overflow)
        if self.intra is not None:
            cols.update(intra_count=self.intra[0], intra_pairs=self.intra[1])
        if self.stepfit is not None:
            cols.update(stepfit_params=self.stepfit.params, stepfit_cost=self.stepfit.cost, stepfit_iters=self.stepfit.iters)
        return cols


class TraceAnalyzer:
    """Stages 1-3 over a time shard with every buffer allocated once and a single host
    synchronisation at the end of the step (the median needs two small ones up front).

    `raw_ext` = [lo_halo | owned | hi_halo] codes.  The filter runs over the extended range
    (its constant pad only matters at the true ends of the trace), and so do the baseline
    blocks and the detector: the state at the first owned sample is then the true one (an
    event in progress at a shard boundary is not seen twice) and an event that starts in the
    owned range and ends in the right halo is completed.  Events are owned by the rank whose
    owned range holds their start.  `lo_halo` must be a multiple of the baseline block so
    that the block grid of every rank is the global one (`required_halo(..., block=)`)."""

    def __init__(self, n_ext: int, settings, cutoff: float, order: int = 8, *, lo_halo: int = 0, hi_halo: int = 0,
                 threshold: float = 5.0, hysteresis: float = 1.0, baseline_block: int = detect.DEFAULT_BASELINE_BLOCK,
                 baseline_min: float, baseline_max: float, padding: int = 1000, event_padding: int = 100,
                 minpoints: int = 8, maxpoints: int = 100_000, cusum_delta: float | None = None,
                 cusum_h: float | None = None, max_levels: int = cusum.DEFAULT_MAX_LEVELS,
                 event_capacity: int | None = None, group=None, device="cuda", fuse_stats: bool = True,
                 fused_count: bool = True, intra_threshold: float = 0.0, intra_hysteresis: float = 0.0,
                 max_crossings: int = 8, halos_clipped_by_trace_ends: bool = False, stepfit_samples: int = 0,
                 stepfit_fallback: bool = False):
        self.n_ext, self.lo_halo, self.hi_halo = int(n_ext), int(lo_halo), int(hi_halo)
        self.n_own = self.n_ext - self.lo_halo - self.hi_halo
        self.n_det = self.n_ext
        if self.lo_halo % int(baseline_block):
            raise ValueError("lo_halo must be a multiple of the baseline block (pipeline.required_halo(..., block=))")
        # a halo (0 = a true end of the trace) must cover the IIR warm-up of both passes and one maximal event window
        need = required_halo(cutoff, order, float(np.floor(np.squeeze(settings["ADCSAMPLERATE"]))),
                             int(maxpoints) + 2 * int(event_padding), int(padding))
        # (`halos_clipped_by_trace_ends`: the caller cut full halos at the true ends of the trace, where nothing is missing)
        for name, h in (("lo_halo", self.lo_halo), ("hi_halo", self.hi_halo)):
            if 0 < h < need and not halos_clipped_by_trace_ends:
                raise ValueError(f"{name} = {h} samples is shorter than the {need} this configuration needs "
                                 "(pipeline.required_halo(cutoff, order, fs, maxpoints + 2 * event_padding))")
        self.settings, self.cutoff, self.order, self.padding = settings, float(cutoff), int(order), int(padding)
        self.threshold, self.hysteresis = float(threshold), float(hysteresis)
        self.block, self.bmin, self.bmax = int(baseline_block), float(baseline_min), float(baseline_max)
        self.event_padding, self.minpoints, self.maxpoints = int(event_padding), int(minpoints), int(maxpoints)
        self.delta, self.h, self.max_levels = cusum_delta, cusum_h, int(max_levels)
        # intra-event threshold crossings (readevents.py:1340-1343, 1363-1367); 0 = off, as in summary.txt
        self.intra_threshold, self.intra_hysteresis = float(intra_threshold), float(intra_hysteresis)
        self.max_crossings = int(max_crossings)
        # step-response fit of the accepted events shorter than `stepfit_samples` (type 1, stepfit.py); 0 = off
        self.stepfit_samples = int(stepfit_samples)
        if self.stepfit_samples < 0:
            raise ValueError("stepfit_samples must be >= 0")
        if self.stepfit_samples and self.stepfit_samples + 2 * self.event_padding > stepfit.MAX_WINDOW:
            raise ValueError(f"stepfit_samples + 2 * event_padding = {self.stepfit_samples + 2 * self.event_padding} exceeds "
                             f"the {stepfit.MAX_WINDOW}-sample window of the step-response fit")
        # the same fit of every event CUSUM+ leaves without a sub-level (type 5 otherwise), whatever its length; with
        # cusum_delta None, of every accepted event
        self.stepfit_fallback = bool(stepfit_fallback)
        if self.stepfit_fallback and self.maxpoints + 2 * self.event_padding > stepfit.LONG_MAX_WINDOW:
            raise ValueError(f"maxpoints + 2 * event_padding = {self.maxpoints + 2 * self.event_padding} exceeds the "
                             f"{stepfit.LONG_MAX_WINDOW}-sample window of the step-response fallback")
        self.fit_on = bool(self.stepfit_samples) or self.stepfit_fallback
        self.tau0 = (stepfit.zero_phase_rise_tau(float(np.floor(np.squeeze(settings["ADCSAMPLERATE"]))), cutoff, order)
                     if self.fit_on else 0.0)
        self.group = group
        self.device = torch.device(device)
        self.mask = filters.chimera_bitmask(settings)
        L = _lib.lib()
        if self.block % L.ct_detect_run():
            raise ValueError(f"baseline block must be a multiple of {L.ct_detect_run()} samples")
        self.y = torch.empty(self.n_ext, dtype=torch.float32, device=self.device)
        self.design = bessel_lowpass(self.order, 2.0 * self.cutoff / float(np.floor(np.squeeze(settings["ADCSAMPLERATE"]))))
        # baseline block sums ride on the filter's epilogue when the block is a whole number of its warp groups
        self.fuse_stats = (bool(fuse_stats) and self.block >= 65536
                           and self.block % filters.stats_granule(self.n_ext, self.padding, self.design) == 0)
        self.fused_count = bool(fused_count)     # the exact-median window tally rides on the forward pass (+0.35 ms against 0.79 ms as its own kernel on C2)
        self.filter_ws = None
        self.minmax = None                         # (min, max) of every 64-sample chunk of y, left by the backward pass
        self.H = max(1, self.design.impulse_tail(filters.DEFAULT_HALO_EPS))
        self.ws_bytes = int(L.ct_detect_workspace_bytes(self.n_det))
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=self.device)
        self._alloc_events(int(event_capacity) if event_capacity else max(1024, self.n_det // 2048))

    def _alloc_events(self, cap: int) -> None:
        dev = self.device
        self.cap = cap
        self.starts = torch.empty(cap, dtype=torch.int64, device=dev)
        self.ends = torch.empty(cap, dtype=torch.int64, device=dev)
        self.w0 = torch.empty(cap, dtype=torch.int64, device=dev)
        self.w1 = torch.empty(cap, dtype=torch.int64, device=dev)
        self.typ = torch.empty(cap, dtype=torch.int32, device=dev)
        self.scalars = torch.zeros(4, dtype=torch.int64, device=dev)     # n_starts, n_ends, n_kept, first kept index
        self.median_result = torch.zeros(4, dtype=torch.int32, device=dev)   # CtMedianResult: code1, code2, pad_x (float bits), status
        self.intra = ((torch.zeros(cap, dtype=torch.int32, device=dev),
                       torch.full((cap, 2 * self.max_crossings), -1, dtype=torch.int32, device=dev))
                      if self.intra_threshold > 0 else None)
        self.levels = cusum.LevelTable.empty(cap, self.max_levels, dev) if self.delta is not None or self.fit_on else None
        if self.stepfit_fallback:
            self.sf_counter = torch.empty(1, dtype=torch.int64, device=dev)     # rows claimed by the long fit
        self.fit = (stepfit.StepFitTable(torch.empty((cap, 6), dtype=torch.float64, device=dev),
                                         torch.empty(cap, dtype=torch.float64, device=dev),
                                         torch.empty(cap, dtype=torch.int32, device=dev), self.typ)
                    if self.fit_on else None)
        if self.delta is not None:
            self.cws_bytes = int(_lib.lib().ct_cusum_workspace_bytes(cap))
            self.cws = torch.empty((self.cws_bytes + 7) // 8, dtype=torch.int64, device=dev)

    def run_from_host(self, host_codes: torch.Tensor, chunks: int = 16, stage_hook=None) -> AnalysisResult:
        """`run` with the codes still in (pinned) host memory: the host->device copy is cut into
        `chunks` pieces on a copy stream and the forward filter pass (with the median count on its
        side) follows the copy chunk by chunk, so only the work after the forward pass is left when the
        last byte arrives.  Possible because the forward pass needs the median only approximately:
        the estimate comes from the first chunk, the exact value from the fused count."""
        if host_codes.numel() != self.n_ext or host_codes.dtype not in (torch.uint16, torch.int16) or host_codes.is_cuda:
            raise ValueError("host_codes must be a CPU uint16/int16 tensor of the planned length")
        if getattr(self, "raw_dev", None) is None:
            self.raw_dev = torch.empty(self.n_ext, dtype=host_codes.dtype, device=self.device)
            self.copy_stream = torch.cuda.Stream(device=self.device)
        gran = 1 << 20
        per = max(gran, -(-self.n_ext // int(chunks) // gran) * gran)
        bounds = list(range(0, self.n_ext, per)) + [self.n_ext]
        events = []
        cur = torch.cuda.current_stream(self.device)
        self.copy_stream.wait_stream(cur)                      # the previous step may still read raw_dev
        with torch.cuda.stream(self.copy_stream):
            for a, b in zip(bounds[:-1], bounds[1:]):
                self.raw_dev[a:b].copy_(host_codes[a:b], non_blocking=True)
                e = torch.cuda.Event()
                e.record(self.copy_stream)
                events.append(e)
        return self.run(self.raw_dev, stage_hook=stage_hook, _arrivals=(bounds, events))

    def run(self, raw_ext: torch.Tensor, stage_hook=None, _arrivals=None, _fixed=None) -> AnalysisResult:
        # the library keys its per-device state on the CURRENT device: make it the tensors' device
        with torch.cuda.device(self.device):
            return self._run(raw_ext, stage_hook, _arrivals, _fixed)

    def _run(self, raw_ext: torch.Tensor, stage_hook=None, _arrivals=None, _fixed=None, _host_median: bool = False) -> AnalysisResult:
        """One pass of stages 1-3.  `stage_hook(name)` (optional) is called after the launches of each
        stage have been enqueued: 'median', 'filter', 'baseline', 'detect', 'cusum' (profiling only).
        `_fixed = (MedianPlan, pad_x, (c1, c2))` (StreamingAnalyzer) skips the median stages: the filter
        subtracts `plan.est` and pads with `pad_x` = median - estimate."""
        hook = stage_hook or (lambda name: None)
        if raw_ext.numel() != self.n_ext:
            raise ValueError(f"analyzer was planned for {self.n_ext} samples, got {raw_ext.numel()}")
        L = _lib.lib()
        lo, n_own = self.lo_halo, self.n_own
        owned = raw_ext[lo:lo + n_own]
        st = filters._stream_ptr(raw_ext)
        cur = torch.cuda.current_stream(self.device)
        # ---- median, phase 1: estimate (subtraction constant of the filter, verification window)
        hist_fn, count_fn = median.device_counters(owned, self.mask)
        if _fixed is not None:
            plan = _fixed[0]
        elif _arrivals is None:
            plan = median.estimate(n_own, self.mask, hist_fn, self.group)
        else:                                                  # only the first chunk has arrived: estimate from it
            bounds, events = _arrivals
            cur.wait_event(events[0])
            first = raw_ext[lo:max(lo + 1, min(bounds[1], lo + n_own))]
            plan = median.estimate(n_own, self.mask, median.device_counters(first, self.mask)[0], self.group,
                                   n_sampled=first.numel())
        hook("median")
        if self.filter_ws is None:
            need = int(L.ct_filtfilt_workspace_bytes(self.n_ext, self.padding, self.H))
            self.filter_ws = torch.empty(need, dtype=torch.uint8, device=self.device)
            self.minmax = torch.empty(2 * int(L.ct_filter_summary_count(self.n_ext, self.padding, self.H)), dtype=torch.float32,
                                      device=self.device)
        coef = filters.make_coef(self.design)
        alpha, _ = filters.chimera_affine(self.settings)
        origin = 0
        # ---- forward pass with the estimate; it tallies the window counts of the owned codes on the side
        route = median.route(plan, fixed=_fixed is not None, streamed=_arrivals is not None, fused_count=self.fused_count)
        plan.lo = route.lo
        counts = torch.zeros(9, dtype=torch.int64, device=self.device) if route.count else None
        pieces = [(0, 0, self.n_ext)] if _arrivals is None else [(2, a, b) for a, b in zip(_arrivals[0][:-1], _arrivals[0][1:])]
        pad_first = float(_fixed[1]) if _fixed is not None else 0.0
        for i, (part, a, b) in enumerate(pieces):
            if _arrivals is not None:
                cur.wait_event(_arrivals[1][i])
            rc = L.ct_filter_forward_u16(raw_ext.data_ptr(), self.n_ext, self.padding, float(plan.est), self.mask, pad_first,
                                         C.byref(coef), self.H, origin, part, plan.lo, plan.step, lo, lo + n_own,
                                         counts.data_ptr() if route.count == "ride" else None, a, b,
                                         self.filter_ws.data_ptr(), self.filter_ws.numel(), st)
            _lib.check(rc, "ct_filter_forward_u16")
            if route.count == "kernel":            # the window count of this piece's owned codes as its own kernel
                median.count_window(raw_ext[max(a, lo):min(b, lo + n_own)], self.mask, plan.lo, plan.step, counts, route.nbins)
        # everything the backward launch needs that does not depend on the exact median is prepared BEFORE the host waits
        # for the counts: the GPU idles from the end of the forward pass to the backward launch
        bl = detect.new_baseline(self.n_det, self.block, self.bmin, self.bmax, self.device) if self.fuse_stats else None
        stats = detect.stats_args(bl, origin=0) if bl is not None else None
        offset = float(filters.scale_codes_host(np.array([plan.est], dtype=np.uint16), self.settings)[0])
        # ---- median, phase 2: exact order statistics
        on_device = route.device and not _host_median
        self.last_median_route = "device" if on_device else ("host after a device miss" if _host_median else "host")
        if on_device:
            # no host round trip between the passes: one thread turns the (summed) counts into the two middle codes and the
            # pad of the filter ends, the end groups re-run with it (their CTAs return at once when the estimate was the
            # median), and the backward pass follows; the codes reach the host with the step's one synchronisation.  If
            # the window missed them (status != 0) the step is redone the host-driven way.
            median.verify_on_device(plan, counts, route.nbins, self.median_result, self.group)
            rc = L.ct_filter_forward_ends_u16(raw_ext.data_ptr(), self.n_ext, self.padding, float(plan.est), self.mask,
                                              self.median_result[2:].data_ptr(), C.byref(coef), self.H, origin,
                                              self.filter_ws.data_ptr(), self.filter_ws.numel(), st)
            _lib.check(rc, "ct_filter_forward_ends_u16")
            c1 = c2 = None
        else:
            if _fixed is not None:
                c1, c2 = _fixed[2]
            else:
                c1, c2 = median.search(n_own, self.mask, hist_fn, count_fn, self.group, plan=plan, first_counts=counts)
            pad_x = 0.5 * (c1 + c2) - plan.est if _fixed is None else 0.0
            if pad_x != 0.0:        # the pad holds median - estimate: redo the groups at the two ends of the trace
                rc = L.ct_filter_forward_u16(raw_ext.data_ptr(), self.n_ext, self.padding, float(plan.est), self.mask,
                                             float(pad_x), C.byref(coef), self.H, origin, 1, 0, 1, 0, 0, None, 0, 0,
                                             self.filter_ws.data_ptr(), self.filter_ws.numel(), st)
                _lib.check(rc, "ct_filter_forward_u16")
        y = self.y
        rc = L.ct_filter_backward(self.n_ext, self.padding, float(plan.est), float(alpha), offset, C.byref(coef), self.H, origin,
                                  y.data_ptr(), self.filter_ws.data_ptr(), self.filter_ws.numel(),
                                  C.byref(stats) if stats is not None else None, self.minmax.data_ptr(), st)
        _lib.check(rc, "ct_filter_backward")
        yd = y
        st = filters._stream_ptr(y)
        hook("filter")
        if bl is not None:
            detect.finish_baseline(bl, self.threshold, self.hysteresis)
        else:
            bl = detect.baseline_blocks(yd, self.block, self.bmin, self.bmax, threshold=self.threshold,
                                        hysteresis=self.hysteresis)
        sign, ts, te = bl.device_lines(self.device)
        hook("baseline")
        while True:
            sc = self.scalars
            rc = L.ct_detect_f32(yd.data_ptr(), self.n_det, self.block, sign.data_ptr(), ts.data_ptr(), te.data_ptr(), 0,
                                 self.minmax.data_ptr(), 0, self.ws.data_ptr(), self.ws_bytes, self.starts.data_ptr(),
                                 self.ends.data_ptr(), self.cap, sc[0:].data_ptr(), st)
            _lib.check(rc, "ct_detect_f32")
            rc = L.ct_event_windows(self.starts.data_ptr(), self.ends.data_ptr(), sc[0:].data_ptr(), self.cap, self.n_det,
                                    lo, lo + n_own, self.event_padding, self.minpoints, self.maxpoints, self.w0.data_ptr(),
                                    self.w1.data_ptr(), self.typ.data_ptr(), sc[2:].data_ptr(), st)
            _lib.check(rc, "ct_event_windows")
            hook("detect")
            if self.stepfit_samples:             # before CUSUM+, which then skips the short events
                stepfit.select_short(self.w0, self.w1, self.typ, padding=self.event_padding,
                                     stepfit_samples=self.stepfit_samples, n_events_dev=sc[2:])
            lv = self.levels
            if self.delta is not None:
                rc = L.ct_cusum_batch_dev(yd.data_ptr(), self.n_det, self.w0.data_ptr(), self.w1.data_ptr(),
                                          self.typ.data_ptr(), sc[2:].data_ptr(), self.cap, float(self.delta),
                                          float(self.h), self.max_levels, lv.n_levels.data_ptr(), lv.edges.data_ptr(),
                                          lv.mean.data_ptr(), lv.std.data_ptr(), lv.overflow.data_ptr(), self.cws.data_ptr(),
                                          self.cws_bytes, st)
                _lib.check(rc, "ct_cusum_batch_dev")
            elif self.fit_on:                    # no CUSUM+: the rows of the events the fit does not take stay empty
                lv.clear()
            if self.stepfit_fallback:            # the events CUSUM+ left without a sub-level: type 1, or 8 (long)
                stepfit.select_fallback(lv, self.w0, self.w1, self.typ, n_events_dev=sc[2:], capacity=self.cap)
            if self.fit_on:                      # after CUSUM+, which writes n_levels = 0 for every event not of type 0
                stepfit.launch(yd, self.w0, self.w1, self.typ, self.fit, lv, padding=self.event_padding, tau0=self.tau0,
                               n_events_dev=sc[2:], capacity=self.cap)
            if self.stepfit_fallback:            # after the short fit, which zeroes the params of every row not of type 1
                stepfit.launch_long(yd, self.w0, self.w1, self.typ, self.fit, lv, padding=self.event_padding,
                                    tau0=self.tau0, n_events_dev=sc[2:], capacity=self.cap, row_counter=self.sf_counter)
            if self.intra is not None:
                # the block of the event start: win_start + padding (windows are compacted, the start list is not)
                detect.intra_crossings(yd, self.w0, self.w1, self.w0 + self.event_padding, bl, self.intra_threshold,
                                       self.intra_hysteresis, max_pairs=self.max_crossings, n_events_dev=sc[2:],
                                       out=self.intra)
            hook("cusum")
            tail = (self.median_result.to(torch.int64),) if on_device else ()
            host = torch.cat((sc[:4], bl.dev["status"].to(torch.int64)) + tail).cpu().numpy()   # the step's one sync
            if on_device:
                if int(host[8]) != 0:                # the four-code window missed the median (every rank sees the same counts)
                    return self._run(raw_ext, stage_hook, _arrivals, _fixed, _host_median=True)
                c1, c2 = int(host[5]), int(host[6])
            ns, ne, nk, i0 = int(host[0]), int(host[1]), int(host[2]), int(host[3])
            if max(ns, ne) <= self.cap:
                break
            self._alloc_events(max(ns, ne))          # more events than planned: grow and redo stages 2-3
        self.last_median = (c1, c2)
        pad_value = float(np.median(filters.scale_codes_host(np.array([c1, c2], dtype=np.uint16), self.settings)))
        status = int(host[4]) != 0
        if _fixed is None:
            # the error decision is collective: the flag rides with the event counts, then every rank raises
            first_id, total, bad = event_ids_and_status(0 if status else nk, int(status), self.group, self.device)
        else:
            first_id, total, bad = 0, nk, int(status)
        if bad:
            raise ValueError("no baseline block has enough samples inside [baseline_min, baseline_max]"
                             + ("" if status else " (on another rank)"))
        bl._checked = True
        open_start = -1
        if ns > ne:                                   # an event still open at the end of the data
            o = int(self.starts[ne].item()) - lo
            open_start = o if 0 <= o < n_own else -1
        # event indices are reported relative to the first owned sample
        ev = detect.EventList(self.starts[i0:i0 + nk] - lo, self.ends[i0:i0 + nk] - lo, open_start)
        return AnalysisResult(filtered=y[lo:lo + n_own], detect_trace=yd, lo_halo=lo, baseline=bl, events=ev,
                              win_start=self.w0[:nk], win_end=self.w1[:nk], types=self.typ[:nk],
                              levels=None if self.levels is None else self.levels.rows(nk),
                              pad_value=pad_value, median_codes=(c1, c2), first_event_id=first_id, total_events=total,
                              intra=None if self.intra is None else (self.intra[0][:nk], self.intra[1][:nk]),
                              stepfit=None if self.fit is None else self.fit.rows(nk))


    def tables_to_host(self, r: AnalysisResult) -> dict:
        """Event and level tables of `r` as numpy arrays: device -> pinned host buffers
        (allocated once at capacity) with one synchronisation; the arrays alias the pinned
        buffers and are valid until the next call."""
        nk = int(r.events.starts.numel())
        if getattr(self, "_pinned_cap", 0) < self.cap:
            self._pinned = {}
            self._pinned_cap = self.cap
        out = {}
        for k, t in r.columns().items():
            if k not in self._pinned:
                self._pinned[k] = torch.empty((self.cap,) + tuple(t.shape[1:]), dtype=t.dtype, pin_memory=True)
            h = self._pinned[k][:nk]
            h.copy_(t, non_blocking=True)
            out[k] = h
        torch.cuda.current_stream(self.device).synchronize()
        return {k: v.numpy() for k, v in out.items()}


@dataclass
class StreamResult:
    """What `StreamingAnalyzer.run_from_host` leaves behind: the filtered trace and the baseline
    table on the device, the event / level tables already in (pinned) host memory."""
    filtered: torch.Tensor          # float32 CUDA, the rank's owned samples
    baseline: detect.Baseline       # blocks of the owned range
    tables: dict                    # numpy: AnalysisResult.columns of the sub-shards, starts / ends from the first owned sample
    pad_value: float
    median_codes: tuple[int, int]
    first_event_id: int = 0
    total_events: int = 0
    redone: str = ""                # "", "first" (first sub-shard redone with the exact pad) or "whole" (fallback)


class _HostFeed:
    """Pieces of a trace that already sits in (pinned) host memory: every copy is queued up front."""

    def __init__(self, host_codes: torch.Tensor):
        self.host = host_codes

    def start(self, an: "StreamingAnalyzer", pieces, cur) -> None:
        self.events = []
        an.copy_stream.wait_stream(cur)                        # the previous step may still read raw_dev
        with torch.cuda.stream(an.copy_stream):
            for a, b in pieces:
                if b > a:
                    an.raw_dev[a:b].copy_(self.host[a:b], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(an.copy_stream)
                self.events.append(ev)

    def wait(self, i: int, cur) -> None:
        cur.wait_event(self.events[i])

    def finish(self) -> None:
        pass

    def whole(self, an: "StreamingAnalyzer") -> torch.Tensor:
        return self.host


class _FileFeed:
    """Pieces read from the `.log` series on a worker thread (loader.WindowReader: several reader threads fill
    disjoint parts of a pinned slab with preadv, GIL released), each handed to the copy engine as soon as it is in
    memory; `slabs` pinned slabs rotate, so reading piece i+1 overlaps the host->device copy of piece i and the
    kernels of piece i-1 (plot-trace.py:230-299 reads the whole window before anything else happens)."""

    def __init__(self, reader, threads: int = 8, slabs: int = 3):
        self.reader, self.threads, self.nslabs = reader, int(threads), int(slabs)
        self.error = None

    def start(self, an: "StreamingAnalyzer", pieces, cur) -> None:
        import threading
        need = max((b - a for a, b in pieces), default=1)
        pool = getattr(an, "_slabs", None)
        if pool is None or len(pool) != self.nslabs or pool[0].numel() < need:
            pool = an._slabs = [torch.empty(need, dtype=an.raw_dev.dtype, pin_memory=True) for _ in range(self.nslabs)]
        self.slabs = pool
        self.ready = [threading.Event() for _ in pieces]
        self.events = [None] * len(pieces)
        an.copy_stream.wait_stream(cur)
        self.thread = threading.Thread(target=self._run, args=(an, list(pieces)), daemon=True)
        self.thread.start()

    def _run(self, an, pieces) -> None:
        from concurrent.futures import ThreadPoolExecutor
        try:
            with torch.cuda.device(an.device), ThreadPoolExecutor(self.threads) as pool:
                slab_ev = [None] * self.nslabs
                for i, (a, b) in enumerate(pieces):
                    j = i % self.nslabs
                    if slab_ev[j] is not None:
                        slab_ev[j].synchronize()               # the slab's previous copy has left host memory
                    if b > a:
                        dst = self.slabs[j].numpy()
                        cuts = np.linspace(a, b, self.threads + 1).astype(np.int64)
                        futs = [pool.submit(self.reader.read_into, dst[int(c0) - a:], int(c0), int(c1))
                                for c0, c1 in zip(cuts[:-1], cuts[1:]) if c1 > c0]
                        for f in futs:
                            f.result()
                    with torch.cuda.stream(an.copy_stream):
                        if b > a:
                            an.raw_dev[a:b].copy_(self.slabs[j][:b - a], non_blocking=True)
                        ev = torch.cuda.Event()
                        ev.record(an.copy_stream)
                    slab_ev[j] = self.events[i] = ev
                    self.ready[i].set()
        except BaseException as e:                              # surfaces in wait()
            self.error = e
            for r in self.ready:
                r.set()

    def wait(self, i: int, cur) -> None:
        self.ready[i].wait()
        if self.error is not None:
            raise self.error
        cur.wait_event(self.events[i])

    def finish(self) -> None:
        self.thread.join()

    def whole(self, an: "StreamingAnalyzer") -> torch.Tensor:
        host = torch.empty(an.n_ext, dtype=an.raw_dev.dtype, pin_memory=True)
        self.reader.read_into(host.numpy(), 0, an.n_ext)
        return host


class StreamingAnalyzer:
    """Stages 1-3 over a trace that is still in pinned host memory, overlapped with its own
    host->device copy: the owned range is cut into time sub-shards (the multi-GPU sharding of
    SURVEY.md 8e applied in sequence on one GPU: halo of `required_halo` samples on each side,
    events owned by the sub-shard that holds their start), the copy is cut at the points where
    a sub-shard becomes complete, and each sub-shard is filtered, detected, segmented and its
    tables are sent back while the next pieces are still arriving.  When the last byte lands only
    the last sub-shard is left to do.

    The exact median (the reference's pad value, plot-trace.py:319) is known only at the end; the
    filter needs it only as the pad at the two true ends of the trace (`filtfilt(code - c) + c`
    does not depend on c otherwise), so every sub-shard subtracts the estimate from the first
    piece, the last one is padded with the exact value, and the (small) first one is redone if the
    estimate turns out to be off.  Interior sub-shard boundaries differ from a whole-trace run only by
    the IIR warm-up error (< 1e-7 of the signal range, as between GPUs).  Blocks without enough
    baseline samples inherit the nearest earlier valid block of their own sub-shard."""

    def __init__(self, n_ext: int, settings, cutoff: float, order: int = 8, *, lo_halo: int = 0, hi_halo: int = 0,
                 shards: int = 16, first_blocks: int = 4, group=None, device="cuda", **kw):
        self.n_ext, self.lo_halo, self.hi_halo = int(n_ext), int(lo_halo), int(hi_halo)
        self.n_own = self.n_ext - self.lo_halo - self.hi_halo
        self.settings, self.cutoff, self.order = settings, float(cutoff), int(order)
        self.group, self.device, self.kw = group, torch.device(device), dict(kw)
        self.block = int(kw.get("baseline_block", detect.DEFAULT_BASELINE_BLOCK))
        self.padding = int(kw.get("padding", 1000))
        self.mask = filters.chimera_bitmask(settings)
        fs = float(np.floor(np.squeeze(settings["ADCSAMPLERATE"])))
        max_event = int(kw.get("maxpoints", 100_000)) + 2 * int(kw.get("event_padding", 100))
        self.h = required_halo(self.cutoff, self.order, fs, max_event, self.padding, block=self.block)
        if self.lo_halo % self.block:
            raise ValueError("lo_halo must be a multiple of the baseline block (pipeline.required_halo(..., block=))")
        a0, b_end = self.lo_halo, self.lo_halo + self.n_own
        cuts = [a0]
        if first_blocks * self.block < self.n_own and shards > 1:
            cuts.append(a0 + first_blocks * self.block)
        per = max(self.block, -(-(b_end - cuts[-1]) // max(1, int(shards)) // self.block) * self.block)
        while cuts[-1] < b_end:
            cuts.append(min(b_end, cuts[-1] + per))
        # (a, b, ea, eb): owned [a, b) and extended [ea, eb) ranges of each sub-shard, in raw_ext coordinates
        self.sub = [(a, b, max(0, a - self.h), min(self.n_ext, b + self.h)) for a, b in zip(cuts[:-1], cuts[1:])]
        self.analyzers: dict = {}
        self.y = torch.empty(self.n_own, dtype=torch.float32, device=self.device)
        self.raw_dev = None
        self.copy_stream = torch.cuda.Stream(device=self.device)
        self.bmin, self.bmax = float(kw["baseline_min"]), float(kw["baseline_max"])
        self._pin, self._pin_cap = {}, 0
        self._whole = None

    # -- helpers -------------------------------------------------------------------
    def _analyzer(self, a, b, ea, eb) -> TraceAnalyzer:
        key = (eb - ea, a - ea, eb - b)
        if key not in self.analyzers:
            self.analyzers[key] = TraceAnalyzer(eb - ea, self.settings, self.cutoff, self.order, lo_halo=a - ea,
                                                hi_halo=eb - b, group=None, device=self.device,
                                                halos_clipped_by_trace_ends=True, **self.kw)
        return self.analyzers[key]

    def _pinned(self, name: str, like: torch.Tensor, rows: int) -> torch.Tensor:
        """Row-capacity-managed pinned host column (grown geometrically, contents kept)."""
        t = self._pin.get(name)
        if t is None or t.shape[0] < rows:
            cap = max(rows, 2 * (t.shape[0] if t is not None else 0), 4096, self.n_own // 2048)
            new = torch.empty((cap,) + tuple(like.shape[1:]), dtype=like.dtype, pin_memory=True)
            if t is not None:
                torch.cuda.current_stream(self.device).synchronize()
                new[:t.shape[0]] = t
            self._pin[name] = t = new
        return t

    def _process(self, i: int, plan: median.MedianPlan, pad_x: float, med: tuple[int, int], row0: int, bl: detect.Baseline,
                 end_at: int | None = None) -> int:
        """Analyse sub-shard i (its data must be resident), store its owned samples, blocks and table rows
        (from row `row0`, or ending at row `end_at`); returns its event count (-1: more rows than `end_at`)."""
        a, b, ea, eb = self.sub[i]
        an = self._analyzer(a, b, ea, eb)
        r = an.run(self.raw_dev[ea:eb], _fixed=(plan, pad_x, med))
        a0 = self.lo_halo
        self.y[a - a0:b - a0].copy_(r.filtered)
        k0, nbk, g0 = (a - ea) // self.block, -(-(b - a) // self.block), (a - a0) // self.block
        for name in ("cnt", "s1", "s2", "mean", "std", "sign", "t_start", "t_end"):
            bl.dev[name][g0:g0 + nbk].copy_(r.baseline.dev[name][k0:k0 + nbk])
        nk = int(r.events.starts.numel())
        if end_at is not None:
            if nk > end_at:
                return -1
            row0 = end_at - nk
        for name, t in r.columns(a - a0).items():
            self._pinned(name, t, row0 + nk)[row0:row0 + nk].copy_(t, non_blocking=True)
        return nk

    def run_from_host(self, host_codes: torch.Tensor) -> StreamResult:
        """`host_codes`: CPU (ideally pinned) uint16/int16 tensor [lo_halo | owned | hi_halo].  One
        host synchronisation per sub-shard (its event count), all hidden under the copy except the last."""
        if host_codes.numel() != self.n_ext or host_codes.dtype not in (torch.uint16, torch.int16) or host_codes.is_cuda:
            raise ValueError("host_codes must be a CPU uint16/int16 tensor of the planned length")
        with torch.cuda.device(self.device):
            return self._run_stream(_HostFeed(host_codes), host_codes.dtype)

    def run_from_file(self, reader, threads: int = 8, slabs: int = 3) -> StreamResult:
        """The same with the codes still in the `.log` files: `reader` = loader.ChimeraSeries(...).reader(start_s,
        end_s) over [lo_halo | owned | hi_halo].  A worker thread reads the pieces into rotating pinned slabs and
        queues their host->device copies; file reads, PCIe and kernels overlap (the from-file path of SURVEY.md 8d/f4)."""
        if int(reader.n) != self.n_ext:
            raise ValueError(f"analyzer was planned for {self.n_ext} samples, the window holds {reader.n}")
        with torch.cuda.device(self.device):
            return self._run_stream(_FileFeed(reader, threads, slabs), torch.uint16)

    def _run_stream(self, feed, dtype) -> StreamResult:
        if self.raw_dev is None or self.raw_dev.dtype != dtype:
            self.raw_dev = torch.empty(self.n_ext, dtype=dtype, device=self.device)
        cur =torch.cuda.current_stream(self.device)
        a0, b_end = self.lo_halo, self.lo_halo + self.n_own
        # ---- the copy, cut where each sub-shard's extended range is complete
        ends = [eb for (_, _, _, eb) in self.sub]
        ends[-1] = self.n_ext
        arrivals, prev = [], 0
        for e in ends:
            arrivals.append((prev, max(prev, e)))
            prev = max(prev, e)
        feed.start(self, arrivals, cur)
        try:
            return self._consume(feed, arrivals, cur, a0, b_end)
        finally:
            feed.finish()

    def _consume(self, feed, arrivals, cur, a0, b_end) -> StreamResult:
        # ---- median estimate from the first piece
        feed.wait(0, cur)
        first = self.raw_dev[a0:max(a0 + 1, min(arrivals[0][1], b_end))]
        plan = median.estimate(self.n_own, self.mask, median.device_counters(first, self.mask)[0], self.group,
                               n_sampled=first.numel())
        self.last_plan = plan
        counts = torch.zeros(9, dtype=torch.int64, device=self.device)
        hist_fn, count_fn = median.device_counters(self.raw_dev[a0:b_end], self.mask)
        bl = detect.new_baseline(self.n_own, self.block, self.bmin, self.bmax, self.device)
        # The first sub-shard holds the true start of the trace, whose pad needs the exact median: it is analysed
        # with the estimate right away and again at the end if the estimate was off.  Its rows sit RIGHT-ALIGNED
        # in a reserved head of the tables, so a different event count the second time moves nothing else.
        head = self.lo_halo == 0 and len(self.sub) > 1
        reserve = max(1024, (self.sub[0][3] - self.sub[0][2]) // 512) if head else 0
        rows, first_rows = reserve, 0
        med, pad_x, redone = (0, 0), 0.0, ""
        # A sub-shard without a single valid baseline block (or more events at the very start than the reserved head
        # holds) sends this rank to the whole-trace analyzer.  That decision must be COLLECTIVE: the rank keeps taking
        # part in the median collectives below, the flag rides with the event counts, and all ranks fall back together.
        failed = False

        def attempt(*args, **kwargs) -> int:
            nonlocal failed
            try:
                return self._process(*args, **kwargs)
            except ValueError as e:
                if "baseline block" not in str(e):
                    raise
                failed = True
                return 0

        for i, (pa, pe) in enumerate(arrivals):
            feed.wait(i, cur)
            if plan.exact is None:                        # exact-median window count of this piece's owned codes
                median.count_window(self.raw_dev[max(pa, a0):min(pe, b_end)], self.mask, plan.lo, plan.step, counts)
            last = i == len(arrivals) - 1
            if last:                                      # everything has arrived: exact order statistics
                med = median.search(self.n_own, self.mask, hist_fn, count_fn, self.group, plan=plan,
                                    first_counts=counts if plan.exact is None else None)
                pad_x = 0.5 * (med[0] + med[1]) - plan.est
            if failed:
                continue
            if head and i == 0:
                first_rows = attempt(0, plan, 0.0, med, 0, bl, end_at=reserve)
            else:
                rows += attempt(i, plan, pad_x if last else 0.0, med, rows, bl)
        if head and not failed and (pad_x != 0.0 or first_rows < 0):
            first_rows = attempt(0, plan, pad_x, med, 0, bl, end_at=reserve)
            redone = "first"
        if first_rows < 0:                                # more events at the very start than the reserved head holds
            failed = True
        start = reserve - max(first_rows, 0)
        first_id, total, any_failed = event_ids_and_status(0 if failed else rows - start, int(failed), self.group, self.device)
        if any_failed:
            return self._run_whole(feed.whole(self))
        cur.synchronize()
        bl.dev["have_thresholds"] = True
        bl._checked = True
        bl.threshold, bl.hysteresis = float(self.kw.get("threshold", 5.0)), float(self.kw.get("hysteresis", 1.0))
        pad_value = float(np.median(filters.scale_codes_host(np.array(med, dtype=np.uint16), self.settings)))
        tables = {k: v[start:rows].numpy() for k, v in self._pin.items()}
        return StreamResult(filtered=self.y, baseline=bl, tables=tables, pad_value=pad_value, median_codes=tuple(med),
                            first_event_id=first_id, total_events=total, redone=redone)

    def _run_whole(self, host_codes: torch.Tensor) -> StreamResult:
        """Fallback: the whole range through one TraceAnalyzer (baseline inheritance across the whole trace)."""
        if self._whole is None:
            self._whole = TraceAnalyzer(self.n_ext, self.settings, self.cutoff, self.order, lo_halo=self.lo_halo,
                                        hi_halo=self.hi_halo, group=self.group, device=self.device, **self.kw)
        r = self._whole.run_from_host(host_codes)
        t = self._whole.tables_to_host(r)
        return StreamResult(filtered=r.filtered, baseline=r.baseline, tables=t, pad_value=r.pad_value,
                            median_codes=r.median_codes, first_event_id=r.first_event_id, total_events=r.total_events,
                            redone="whole")


def analyze_shard(raw_ext: torch.Tensor, settings, cutoff: float, order: int, *, lo_halo: int, hi_halo: int,
                  threshold: float, hysteresis: float, baseline_block: int, baseline_min: float,
                  baseline_max: float, group=None, is_first: bool = True, is_last: bool = True,
                  padding: int = 1000, keep_filtered: bool = True) -> TraceResult:
    """Run stages 1-2 on a time shard (see TraceAnalyzer; this is the one-shot form)."""
    an = TraceAnalyzer(raw_ext.numel(), settings, cutoff, order, lo_halo=lo_halo, hi_halo=hi_halo, threshold=threshold,
                       hysteresis=hysteresis, baseline_block=baseline_block, baseline_min=baseline_min,
                       baseline_max=baseline_max, padding=padding, group=group, device=raw_ext.device)
    r = an.run(raw_ext)
    return TraceResult(filtered=r.filtered if keep_filtered else r.filtered[:0], baseline=r.baseline, events=r.events,
                       pad_value=r.pad_value, median_codes=r.median_codes, first_event_id=r.first_event_id,
                       total_events=r.total_events)


def analyze_trace(raw: torch.Tensor, settings, cutoff: float, order: int = 8, *, threshold: float = 5.0,
                  hysteresis: float = 1.0, baseline_block: int = detect.DEFAULT_BASELINE_BLOCK,
                  baseline_min: float, baseline_max: float, padding: int = 1000) -> TraceResult:
    """Single-GPU stages 1-2 over a whole device-resident trace."""
    return analyze_shard(raw, settings, cutoff, order, lo_halo=0, hi_halo=0, threshold=threshold,
                         hysteresis=hysteresis, baseline_block=baseline_block, baseline_min=baseline_min,
                         baseline_max=baseline_max, padding=padding)


def gather_tables(tables: dict, group=None, dst: int = 0) -> dict | None:
    """Gather per-rank event-table columns (tensors whose first dimension is the rank's event count) to rank
    `dst` in rank order = time order (the one data-sized collective of the path, O(events); SURVEY.md 8e).
    One small all_reduce exchanges the row counts; every column then travels point to point, exactly its rows,
    straight into its slice of the concatenated column on `dst` (one batched send/receive group, no padding and
    nothing sent to ranks that do not need it).  Returns the concatenated columns on `dst`, None elsewhere; with
    `group=None` the input itself."""
    if group is None:
        return tables
    import torch.distributed as dist
    ws, rk = dist.get_world_size(group), dist.get_rank(group)
    first = next(iter(tables.values()))
    dev = first.device
    counts = torch.zeros(ws, dtype=torch.int64, device=dev)
    counts[rk] = first.shape[0]
    counts = _all_reduce_(counts, group).cpu().numpy()
    offs = np.concatenate(([0], np.cumsum(counts)))
    out, ops = {}, []
    for name, t in tables.items():                       # same column order on every rank (dict order)
        t = t.contiguous()
        if rk == dst:
            full = torch.empty((int(offs[-1]),) + tuple(t.shape[1:]), dtype=t.dtype, device=dev)
            full[int(offs[rk]):int(offs[rk + 1])] = t
            for src in range(ws):
                if src != dst and counts[src]:
                    ops.append(dist.P2POp(dist.irecv, full[int(offs[src]):int(offs[src + 1])], dist.get_global_rank(group, src), group))
            out[name] = full
        elif counts[rk]:
            ops.append(dist.P2POp(dist.isend, t, dist.get_global_rank(group, dst), group))
    if ops:
        for w in dist.batch_isend_irecv(ops):
            w.wait()
    return out if rk == dst else None


def shard_bounds(n: int, world: int, rank: int, align: int) -> tuple[int, int]:
    """Owned range of `rank`: equal shares rounded to `align` (the baseline block), so
    baseline blocks never straddle ranks."""
    per = -(-n // world)
    per = -(-per // align) * align
    return min(n, rank * per), min(n, (rank + 1) * per)
