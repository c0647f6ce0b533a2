"""Stage 2 of the hot path: baseline block statistics and threshold/hysteresis event
detection with stream compaction, on the GPU.

The reference contains no implementation of this stage; it draws and consumes its output
(`plot-trace.py:172-203,350-414`: baseline.csv rows `time_s, baseline_pA, stdev_pA`, start
line `baseline - sign*threshold*stdev`, end line `baseline - sign*(threshold-hysteresis)*
stdev`; rate.csv rows `id, type, start_time_s, end_time_s`).  Definition of record:
oracle/events_oracle.py.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from .filters import _require_cuda, _stream_ptr

STATS_MAX_SHIFT = 8
DEFAULT_BASELINE_BLOCK = 1 << 20


def stats_shift(half_width: float, block: int) -> int:
    """Fixed-point fraction bits of the block sums: largest s <= 8 with
    (half_width*2^s + 1)^2 * block < 2^62."""
    s = STATS_MAX_SHIFT
    while s > -32 and (float(half_width) * 2.0 ** s + 1.0) ** 2 * float(block) >= 2.0 ** 62:
        s -= 1
    return s


def check_hysteresis(name: str, value) -> None:
    """Raise ValueError unless `value` >= 0: the end line must lie between the start line and the baseline."""
    if not float(value) >= 0.0:
        raise ValueError(f"{name} must be >= 0, got {value} (a negative hysteresis crosses the start and end lines)")


class Baseline:
    """Per-block baseline table (the rows of baseline.csv) plus the float32 lines the
    detector compares against.  When produced by `baseline_blocks` everything lives on the
    device (`dev` holds the tensors the detector reads) and the numpy views are fetched on
    first access; a table can also be built from host arrays (tests, restored tables)."""

    def __init__(self, block: int, mean=None, std=None, count=None, sign=None, t_start=None, t_end=None, dev=None):
        self.block = int(block)
        self._mean, self._std, self._count = mean, std, count
        self._sign, self._t_start, self._t_end = sign, t_start, t_end
        self.dev = dev              # dict of device tensors: cnt s1 s2 mean std sign t_start t_end status (+ c0, shift)
        self._checked = False

    # -- host views ----------------------------------------------------------------
    def _fetch(self, name):
        self.check()
        return self.dev[name].cpu().numpy()

    def check(self) -> None:
        """Raise if no block had enough samples inside the baseline window (one device read)."""
        if self.dev is not None and not self._checked:
            if int(self.dev["status"].item()) != 0:
                raise ValueError("no baseline block has enough samples inside [baseline_min, baseline_max]")
            self._checked = True

    @property
    def mean(self):
        if self._mean is None:
            self._mean = self._fetch("mean")
        return self._mean

    @property
    def std(self):
        if self._std is None:
            self._std = self._fetch("std")
        return self._std

    @property
    def count(self):
        if self._count is None:
            self._count = self._fetch("cnt")
        return self._count

    def _line(self, name):
        v = getattr(self, "_" + name)
        if v is None and self.dev is not None and self.dev.get("have_thresholds"):
            v = self._fetch(name)
            setattr(self, "_" + name, v)
        return v

    sign = property(lambda self: self._line("sign"), lambda self, v: setattr(self, "_sign", v))
    t_start = property(lambda self: self._line("t_start"), lambda self, v: setattr(self, "_t_start", v))
    t_end = property(lambda self: self._line("t_end"), lambda self, v: setattr(self, "_t_end", v))

    def __len__(self):
        return int(self.dev["mean"].numel()) if self.dev is not None else len(self._mean)

    def with_thresholds(self, threshold: float, hysteresis: float) -> "Baseline":
        """plot-trace.py:408-411: start line = baseline - sign*threshold*stdev, end line =
        baseline - sign*(threshold - hysteresis)*stdev, rounded to float32.  `hysteresis` must be
        >= 0: a negative one puts the end line beyond the start line, where the detector's
        definition no longer holds."""
        check_hysteresis("hysteresis", hysteresis)
        self.threshold, self.hysteresis = float(threshold), float(hysteresis)
        if self.dev is not None:
            d = self.dev
            nb = d["mean"].numel()
            rc = _lib.lib().ct_baseline_finalize(d["cnt"].data_ptr(), d["s1"].data_ptr(), d["s2"].data_ptr(), nb,
                                                 float(d["c0"]), int(d["shift"]), int(d["min_count"]), float(threshold),
                                                 float(hysteresis), d["mean"].data_ptr(), d["std"].data_ptr(),
                                                 d["sign"].data_ptr(), d["t_start"].data_ptr(), d["t_end"].data_ptr(),
                                                 d["status"].data_ptr(), _stream_ptr(d["mean"]))
            _lib.check(rc, "ct_baseline_finalize")
            d["have_thresholds"] = True
            self._sign = self._t_start = self._t_end = None
            return self
        sign = np.where(self._mean >= 0, 1, -1).astype(np.int32)
        self._sign = sign
        self._t_start = (self._mean - sign * threshold * self._std).astype(np.float32)
        self._t_end = (self._mean - sign * (threshold - hysteresis) * self._std).astype(np.float32)
        return self

    def device_lines(self, device):
        """(sign int32, t_start float32, t_end float32) device tensors for the detector."""
        if self.dev is not None and self.dev.get("have_thresholds"):
            return self.dev["sign"], self.dev["t_start"], self.dev["t_end"]
        if self._t_start is None:
            raise ValueError("call Baseline.with_thresholds(threshold, hysteresis) first")
        return (torch.from_numpy(np.ascontiguousarray(self._sign, np.int32)).to(device),
                torch.from_numpy(np.ascontiguousarray(self._t_start, np.float32)).to(device),
                torch.from_numpy(np.ascontiguousarray(self._t_end, np.float32)).to(device))


def lines_for(bl: Baseline, threshold: float, hysteresis: float):
    """(sign, t_start, t_end) device tensors for ANOTHER pair of thresholds over the same block sums
    (the intra-event lines), leaving the table's own detector lines untouched."""
    d = bl.dev
    if d is None:
        raise ValueError("lines_for needs a device-resident baseline table")
    nb = d["mean"].numel()
    dev = d["mean"].device
    f64 = torch.empty((2, max(nb, 1)), dtype=torch.float64, device=dev)
    lines = torch.empty((2, max(nb, 1)), dtype=torch.float32, device=dev)
    sign = torch.empty(max(nb, 1), dtype=torch.int32, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    rc = _lib.lib().ct_baseline_finalize(d["cnt"].data_ptr(), d["s1"].data_ptr(), d["s2"].data_ptr(), nb, float(d["c0"]),
                                         int(d["shift"]), int(d["min_count"]), float(threshold), float(hysteresis),
                                         f64[0].data_ptr(), f64[1].data_ptr(), sign.data_ptr(), lines[0].data_ptr(),
                                         lines[1].data_ptr(), status.data_ptr(), _stream_ptr(d["mean"]))
    _lib.check(rc, "ct_baseline_finalize")
    return sign[:nb], lines[0, :nb], lines[1, :nb]


def intra_crossings(y: torch.Tensor, win_start: torch.Tensor, win_end: torch.Tensor, ev_start: torch.Tensor, bl: Baseline,
                    intra_threshold: float, intra_hysteresis: float, *, max_pairs: int = 8, n_events_dev=None,
                    out=None):
    """Intra-event threshold crossings of every event window (oracle/events_oracle.py::intra_crossings;
    readevents.py:1340-1343,1363-1367): (count int32 [E], pairs int32 [E, 2*max_pairs]) device tensors,
    pairs relative to the window start, valid for k < min(count, max_pairs).  `ev_start` (same coordinates
    as the windows) selects the baseline block whose mean/std define the lines.  `n_events_dev`: event
    count still on the device (rows beyond it are not written); `out`: preallocated (count, pairs)."""
    E = int(win_start.numel())
    dev = y.device
    sign, ts, te = lines_for(bl, intra_threshold, intra_hysteresis)
    if out is None:
        count = torch.zeros(E, dtype=torch.int32, device=dev)
        pairs = torch.full((E, 2 * int(max_pairs)), -1, dtype=torch.int32, device=dev)
    else:
        count, pairs = out
    if E:
        rc = _lib.lib().ct_intra_crossings_f32(y.data_ptr(), y.numel(), win_start.data_ptr(), win_end.data_ptr(),
                                               ev_start.data_ptr(), E, n_events_dev.data_ptr() if n_events_dev is not None else None,
                                               bl.block, len(bl), sign.data_ptr(), ts.data_ptr(), te.data_ptr(), int(max_pairs),
                                               count.data_ptr(), pairs.data_ptr(), _stream_ptr(y))
        _lib.check(rc, "ct_intra_crossings_f32")
    return count, pairs


def new_baseline(n: int, block: int, baseline_min: float, baseline_max: float, device, min_count: int = 16) -> Baseline:
    """An empty device-resident baseline table for a trace of `n` samples; the block sums are
    filled either by `baseline_blocks` (own kernel) or by the filter (`stats_args`)."""
    block = int(block)
    nb = (int(n) + block - 1) // block
    c0 = np.float32(0.5 * (np.float32(baseline_min) + np.float32(baseline_max)))
    hw = max(float(c0) - float(np.float32(baseline_min)), float(np.float32(baseline_max)) - float(c0))
    shift = stats_shift(hw, block)
    m = max(nb, 1)
    acc = torch.empty((3, m), dtype=torch.int64, device=device)
    f64 = torch.empty((2, m), dtype=torch.float64, device=device)
    lines = torch.empty((2, m), dtype=torch.float32, device=device)
    d = {"cnt": acc[0, :nb], "s1": acc[1, :nb], "s2": acc[2, :nb], "mean": f64[0, :nb], "std": f64[1, :nb],
         "sign": torch.empty(m, dtype=torch.int32, device=device)[:nb], "t_start": lines[0, :nb], "t_end": lines[1, :nb],
         "status": torch.zeros(1, dtype=torch.int32, device=device), "c0": float(c0), "shift": shift,
         "min_count": int(min_count), "have_thresholds": False, "bmin": float(baseline_min), "bmax": float(baseline_max)}
    return Baseline(block, dev=d)


def stats_args(bl: Baseline, origin: int = 0) -> "_lib.CtFilterStats":
    """The filter-side description of `bl`'s block sums (ct_filtfilt_u16 `stats`): blocks are
    counted from output sample `origin`."""
    d = bl.dev
    return _lib.CtFilterStats(int(origin), bl.block, d["bmin"], d["bmax"], d["c0"], d["shift"],
                              d["cnt"].data_ptr(), d["s1"].data_ptr(), d["s2"].data_ptr())


def baseline_blocks(y: torch.Tensor, block: int, baseline_min: float, baseline_max: float,
                    min_count: int = 16, *, threshold: float | None = None, hysteresis: float | None = None) -> Baseline:
    """Mean / population std of the samples inside [baseline_min, baseline_max] for every
    block of `block` samples.  The device produces exact integer sums and turns them into
    the table (and, if `threshold` is given, the detector's lines) without a host round
    trip; the arithmetic is oracle/events_oracle.py::baseline_from_stats, operation for
    operation."""
    _require_cuda(y, "y", torch.float32)
    n = y.numel()
    bl = new_baseline(n, block, baseline_min, baseline_max, y.device, min_count)
    d = bl.dev
    rc = _lib.lib().ct_block_stats_f32(y.data_ptr(), n, bl.block, d["bmin"], d["bmax"], d["c0"], d["shift"],
                                       d["cnt"].data_ptr(), d["s1"].data_ptr(), d["s2"].data_ptr(), _stream_ptr(y))
    _lib.check(rc, "ct_block_stats_f32")
    return finish_baseline(bl, threshold, hysteresis)


def finish_baseline(bl: Baseline, threshold: float | None = None, hysteresis: float | None = None) -> Baseline:
    """Block sums -> table (+ detector lines when `threshold` is given), on the device."""
    thr = float("nan") if threshold is None else float(threshold)
    hys = 0.0 if hysteresis is None else float(hysteresis)
    bl.with_thresholds(thr, hys)
    bl.dev["have_thresholds"] = threshold is not None
    return bl


@dataclass
class EventList:
    starts: torch.Tensor      # int64 [E] device, first sample beyond the start line
    ends: torch.Tensor        # int64 [E] device, first sample back beyond the end line
    open_start: int           # start of an event still open at the end of the data, or -1

    def __len__(self) -> int:
        return int(self.starts.numel())


def detect_events(y: torch.Tensor, baseline: Baseline, *, state_in: bool = False,
                  capacity: int | None = None, chunk_minmax: torch.Tensor | None = None, minmax_shift: int = 0) -> EventList:
    """Threshold/hysteresis detection over the whole filtered trace `y` (device float32).
    Event i occupies samples [starts[i], ends[i]).  `chunk_minmax`: the (min, max) pairs of the
    64-sample chunks of `y` the filter's backward pass left (same result, 1/32 of the traffic)."""
    _require_cuda(y, "y", torch.float32)
    L = _lib.lib()
    n = y.numel()
    run = L.ct_detect_run()
    if baseline.block % run:
        raise ValueError(f"baseline block must be a multiple of {run} samples")
    dev = y.device
    sign, ts, te = baseline.device_lines(dev)
    wsb = int(L.ct_detect_workspace_bytes(n))
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    cap = int(capacity) if capacity else max(1024, n // 2048)
    while True:
        starts = torch.empty(cap, dtype=torch.int64, device=dev)
        ends = torch.empty(cap, dtype=torch.int64, device=dev)
        counts = torch.zeros(2, dtype=torch.int64, device=dev)
        with torch.cuda.device(dev):
            rc = L.ct_detect_f32(y.data_ptr(), n, baseline.block, sign.data_ptr(), ts.data_ptr(), te.data_ptr(),
                                 int(bool(state_in)), chunk_minmax.data_ptr() if chunk_minmax is not None else None,
                                 int(minmax_shift), ws.data_ptr(), wsb, starts.data_ptr(), ends.data_ptr(), cap,
                                 counts.data_ptr(), _stream_ptr(y))
        _lib.check(rc, "ct_detect_f32")
        ns, ne = (int(v) for v in counts.cpu().numpy())
        if max(ns, ne) <= cap:
            break
        cap = max(ns, ne)
    starts, ends = starts[:ns], ends[:ne]
    if state_in and ne and (ns == 0 or ne > ns or int(ends[0]) < int(starts[0])):
        ends = ends[1:]          # closes an event opened before this data
        ne -= 1
    open_start = -1
    if ns > ne:
        open_start = int(starts[ne])
        starts = starts[:ne]
    return EventList(starts=starts, ends=ends, open_start=open_start)


def event_windows(starts: torch.Tensor, ends: torch.Tensor, n: int, padding: int, minpoints: int,
                  maxpoints: int):
    """Sample windows [start - padding, end + padding) handed to CUSUM+ and the rate.csv
    `type` code: 0 accepted, 2 too short, 3 too long, 4 padding leaves the trace or overlaps
    a neighbouring event (plot-trace.py:354-357 treats type > 1 as rejected)."""
    w0 = starts - padding
    w1 = ends + padding
    length = ends - starts
    z = torch.zeros(1, dtype=torch.int64, device=starts.device)
    nn = torch.full((1,), n, dtype=torch.int64, device=starts.device)
    prev_end = torch.cat((z, ends[:-1]))
    next_start = torch.cat((starts[1:], nn))
    typ = torch.zeros_like(starts, dtype=torch.int32)
    typ[(w0 < prev_end) | (w1 > next_start) | (w0 < 0) | (w1 > n)] = 4
    typ[length > maxpoints] = 3
    typ[length < minpoints] = 2
    return w0, w1, typ
