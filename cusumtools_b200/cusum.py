"""Stage 3 of the hot path: batched per-event CUSUM+ level segmentation (GPU).

The reference has no implementation (it consumes `level_current_pA`, `level_duration_us`,
`blockages_pA`, `stdev_pA`, `n_levels`: readevents.py:843-846,1297-1306); definition of
record: oracle/events_oracle.py (cusum_event / level_stats)."""
from __future__ import annotations

from dataclasses import dataclass, fields

import numpy as np
import torch

from . import _lib
from .filters import _require_cuda, _stream_ptr

DEFAULT_MAX_LEVELS = 16


@dataclass
class LevelTable:
    """Per-event level fit.  Level i of event e covers window samples
    [edges[e, i], edges[e, i+1]); the first and last level are the baseline padding before
    and after the event (the convention of the ';'-lists in events.csv, readevents.py:844)."""
    n_levels: torch.Tensor     # int32 [E]
    edges: torch.Tensor        # int32 [E, max_levels + 1], unused entries -1
    mean: torch.Tensor         # float64 [E, max_levels]  level current, pA
    std: torch.Tensor          # float64 [E, max_levels]  population standard deviation, pA
    overflow: torch.Tensor     # uint8 [E]  1 = more jumps than max_levels - 1
    max_levels: int

    @classmethod
    def empty(cls, rows: int, max_levels: int, device) -> LevelTable:
        """Uninitialised buffers for `rows` events."""
        return cls(torch.empty(rows, dtype=torch.int32, device=device),
                   torch.empty((rows, max_levels + 1), dtype=torch.int32, device=device),
                   torch.empty((rows, max_levels), dtype=torch.float64, device=device),
                   torch.empty((rows, max_levels), dtype=torch.float64, device=device),
                   torch.empty(rows, dtype=torch.uint8, device=device), int(max_levels))

    @classmethod
    def from_columns(cls, cols: dict, device) -> LevelTable:
        """The level rows of host event-table columns (pipeline.AnalysisResult.columns: named as the fields) on `device`."""
        t = [torch.from_numpy(np.ascontiguousarray(cols[f.name])).to(device) for f in fields(cls)[:5]]
        return cls(*t, int(t[2].shape[1]))         # mean: [E, max_levels]

    def rows(self, n: int) -> LevelTable:
        """The first `n` rows, as views of these buffers."""
        return LevelTable(*(getattr(self, f.name)[:n] for f in fields(self)[:5]), self.max_levels)

    def clear(self) -> None:
        """Every row without levels: n_levels 0, no overflow, edges -1 (mean and std are left as they are)."""
        self.n_levels.zero_(); self.overflow.zero_(); self.edges.fill_(-1)


def cusum_levels(y: torch.Tensor, win_start: torch.Tensor, win_end: torch.Tensor, *, delta: float, h: float,
                 max_levels: int = DEFAULT_MAX_LEVELS, types: torch.Tensor | None = None) -> LevelTable:
    """CUSUM+ segmentation of every event window y[win_start[e]:win_end[e]] (device int64
    index tensors), one warp per event.  `delta` is the expected jump size in pA, `h` the
    log-likelihood threshold; events whose `types` entry is non-zero are skipped."""
    _require_cuda(y, "y", torch.float32)
    _require_cuda(win_start, "win_start", torch.int64)
    _require_cuda(win_end, "win_end", torch.int64)
    E = win_start.numel()
    if win_end.numel() != E:
        raise ValueError("win_start and win_end differ in length")
    dev = y.device
    if types is not None:
        _require_cuda(types, "types", torch.int32)
    lv = LevelTable.empty(E, max_levels, dev)
    for t in (lv.n_levels, lv.mean, lv.std, lv.overflow):     # ct_cusum_batch writes every edges row
        t.zero_()
    L = _lib.lib()
    wsb = int(L.ct_cusum_workspace_bytes(E))
    ws = torch.empty((wsb + 7) // 8, dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):        # the library launches on the current device
        rc = L.ct_cusum_batch(y.data_ptr(), y.numel(), win_start.data_ptr(), win_end.data_ptr(),
                              types.data_ptr() if types is not None else None, E, float(delta), float(h),
                              lv.max_levels, lv.n_levels.data_ptr(), lv.edges.data_ptr(), lv.mean.data_ptr(),
                              lv.std.data_ptr(), lv.overflow.data_ptr(), ws.data_ptr(), wsb, _stream_ptr(y))
    _lib.check(rc, "ct_cusum_batch")
    return lv


def cusum_flat(samples: torch.Tensor, offsets: torch.Tensor, **kw) -> LevelTable:
    """Pre-extracted events in one flat buffer (config C3): event e is
    samples[offsets[e]:offsets[e+1]]."""
    _require_cuda(offsets, "offsets", torch.int64)
    return cusum_levels(samples, offsets[:-1].contiguous(), offsets[1:].contiguous(), **kw)
