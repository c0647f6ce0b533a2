"""The event table and the analysis directory the reference's consumers read.

`readevents.py:1527-1544` opens `events.csv` (+ `rate.csv`, `summary.txt`, `events/`) and
`plot-trace.py:172-203` opens `rate.csv`, `baseline.csv`, `summary.txt`; the reference
contains no producer of these files except `mosaicConverter.py:38-194`, which is therefore
the in-repo definition of every column (names, units, `%.16g;` list format).  Conventions
fixed here (SURVEY.md Appendix A.4 lists the open points):

* the CUSUM+ window of an event is [start - padding, end + padding); its first and last
  level are the baseline before / after the event, so the four list columns carry them as
  first and last entry, as the consumers expect (`readevents.py:844,1300-1302`);
* `effective_baseline_pA` = mean of the two; a blockage is `sign(baseline) * (baseline -
  level)`, positive when the current magnitude drops; `blockages_pA` = [before - eff] +
  sub-level blockages + [after - eff] (`mosaicConverter.py:131-132`);
* `n_levels` = number of sub-levels + 1 (`mosaicConverter.py:79`);
* in-event statistics (`average_blockage_pA`, `area_pC`) run over the sub-levels, i.e. from
  the first to the last changepoint; `area_pC` = average blockage (pA) x that duration (s);
* `residual_pA` = rms of trace minus step fit over the whole window = sqrt(sum len*std^2 / sum len);
* `max_deviation_pA` = largest |sample - effective baseline| in the window;
* `type`: 0 accepted (CUSUM fit; 3-column event file), 1 step-response fit (4-column event file
  `time_us,current_pA,cusum_fit,stepfit`, readevents.py:1334-1337), 2 too short, 3 too long, 4 padding
  overlaps a neighbour or leaves the trace, 5 CUSUM+ found no sub-level, 6 more levels than
  the table holds, 7 step fit failed; types > 1 appear in rate.csv only (`plot-trace.py:354-357`);
  type 1 is a short event (`stepfit_samples`) or, with `stepfit_fallback`, an event CUSUM+ left without a
  sub-level (type 5 without it), of any accepted length; type 7 may then be an event of any length;
* a type-1 event has three level rows from its fit p = (i0, a, u1, u2, tau1, tau2) (stepfit.py):
  edges [0, ceil u1, ceil u2, n], means [i0, i0 - a, i0], std = rms of trace minus fitted step response
  over each; the derived columns follow from them as for a CUSUM fit.  `rc_const1_us` / `rc_const2_us`
  are tau1 / tau2 in us (0 for type 0);
* intra-event threshold crossings (`intra_crossings`, rate.csv `intra_crossing_times_us`) are
  produced when the analyzer is given `intra_threshold` > 0 (detect.intra_crossings; the lines the
  consumer draws at readevents.py:1363-1366); at most `max_crossings` pairs are listed per event,
  the count is complete.

The derived per-event statistics (baselines, blockages, area, residual, max deviation, final type) are computed on
the device, one thread per event from the level table (ct_event_columns, after ct_event_extrema_f32); this module
formats them.  Callers that only have host arrays (tests, converters) get the same columns from the NumPy statement
of the definition in `event_columns_host`.  List columns are kept as padded 2-D arrays (`RaggedColumn`) and turned
into `%.16g;` strings column by column when a file is written: no per-event Python loop anywhere.
"""
from __future__ import annotations

import os
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib, cusum
from .filters import _require_cuda, _stream_ptr

EVENT_COLUMNS = ["id", "type", "start_time_s", "event_delay_s", "duration_us", "threshold", "baseline_before_pA",
                 "baseline_after_pA", "effective_baseline_pA", "area_pC", "average_blockage_pA",
                 "relative_average_blockage", "max_blockage_pA", "relative_max_blockage", "max_blockage_duration_us",
                 "n_levels", "intra_crossings", "rc_const1_us", "rc_const2_us", "residual_pA", "max_deviation_pA",
                 "min_blockage_pA", "relative_min_blockage", "min_blockage_duration_us", "level_current_pA",
                 "level_duration_us", "blockages_pA", "stdev_pA"]
RATE_COLUMNS = ["id", "type", "start_time_s", "end_time_s", "intra_crossing_times_us", "local_stdev", "local_baseline"]
TYPE_STEPFIT, TYPE_NO_SUBLEVEL, TYPE_LEVEL_OVERFLOW, TYPE_STEPFIT_FAILED = 1, 5, 6, 7
GOOD_TYPES = (0, TYPE_STEPFIT)     # the types plot-trace.py:354-357 counts as good events (events.csv rows)


def event_extrema(y: torch.Tensor, win_start: torch.Tensor, win_end: torch.Tensor):
    """(min, max) sample of every event window, float32 device tensors."""
    _require_cuda(y, "y", torch.float32)
    _require_cuda(win_start, "win_start", torch.int64)
    _require_cuda(win_end, "win_end", torch.int64)
    E = win_start.numel()
    lo = torch.empty(E, dtype=torch.float32, device=y.device)
    hi = torch.empty(E, dtype=torch.float32, device=y.device)
    rc = _lib.lib().ct_event_extrema_f32(y.data_ptr(), y.numel(), win_start.data_ptr(), win_end.data_ptr(), E, None,
                                         lo.data_ptr(), hi.data_ptr(), _stream_ptr(y))
    _lib.check(rc, "ct_event_extrema_f32")
    return lo, hi


def event_columns(levels, types, xmin: torch.Tensor, xmax: torch.Tensor, n_events_dev=None):
    """Device side of the derived columns: (cols float64 [E, 12], type int32 [E]) CUDA tensors from a
    `cusum.LevelTable` (+ rate.csv type codes, per-event extrema); see ct_event_columns in the C header."""
    E = int(levels.n_levels.numel())
    dev = levels.n_levels.device
    cols = torch.empty((E, 12), dtype=torch.float64, device=dev)
    tout = torch.empty(E, dtype=torch.int32, device=dev)
    if E:
        with torch.cuda.device(dev):
            rc = _lib.lib().ct_event_columns(levels.n_levels.data_ptr(), levels.edges.data_ptr(), levels.mean.data_ptr(),
                                             levels.std.data_ptr(), types.data_ptr() if types is not None else None,
                                             levels.overflow.data_ptr(), xmin.data_ptr(), xmax.data_ptr(), E,
                                             n_events_dev.data_ptr() if n_events_dev is not None else None,
                                             int(levels.max_levels), cols.data_ptr(), tout.data_ptr(), _stream_ptr(cols))
        _lib.check(rc, "ct_event_columns")
    return cols, tout


def event_columns_host(types, n_levels, edges, level_mean, level_std, overflow, xmin, xmax):
    """NumPy statement of ct_event_columns (same conventions, same level-by-level summation order): the definition
    for callers without device tensors, and what the GPU test compares the kernel with."""
    types = np.asarray(types, np.int32).copy()
    nl = np.asarray(n_levels, np.int64)
    E = nl.size
    edges = np.asarray(edges, np.int64).reshape(E, -1)
    mu = np.asarray(level_mean, np.float64).reshape(E, -1)
    sd = np.asarray(level_std, np.float64).reshape(E, -1)
    ML = mu.shape[1] if E else 0
    types[np.isin(types, GOOD_TYPES) & (np.asarray(overflow) != 0)] = TYPE_LEVEL_OVERFLOW
    types[np.isin(types, GOOD_TYPES) & (nl < 3)] = TYPE_NO_SUBLEVEL
    cols = np.zeros((E, 12))
    ok = np.isin(types, GOOD_TYPES)
    rows = np.nonzero(ok)[0]
    if rows.size:
        L = nl[rows]
        before, after = mu[rows, 0], mu[rows, L - 1]
        eff = 0.5 * (before + after)
        sgn = np.where(eff >= 0, 1.0, -1.0)
        tot = np.zeros(rows.size); res = np.zeros(rows.size); dur = np.zeros(rows.size); wsum = np.zeros(rows.size)
        bmax = np.full(rows.size, -np.inf); bmin = np.full(rows.size, np.inf)
        lmax = np.zeros(rows.size); lmin = np.zeros(rows.size)
        for k in range(ML):                              # level by level, the kernel's order
            valid = k < L
            length = np.where(valid, edges[rows, k + 1] - edges[rows, k], 0).astype(np.float64)
            m, s_ = np.where(valid, mu[rows, k], 0.0), np.where(valid, sd[rows, k], 0.0)
            tot = tot + length
            res = res + length * s_ * s_
            inner = valid & (k >= 1) & (k < L - 1)
            dur = np.where(inner, dur + length, dur)
            wsum = np.where(inner, wsum + length * m, wsum)
            b = sgn * (eff - m)
            up, dn = inner & (b > bmax), inner & (b < bmin)
            bmax, lmax = np.where(up, b, bmax), np.where(up, length, lmax)
            bmin, lmin = np.where(dn, b, bmin), np.where(dn, length, lmin)
        with np.errstate(invalid="ignore", divide="ignore"):
            avg = sgn * (eff - wsum / dur)
            resid = np.sqrt(res / tot)
        xm, xM = np.asarray(xmin, np.float64)[rows], np.asarray(xmax, np.float64)[rows]
        dev_ = np.maximum(np.abs(xM - eff), np.abs(xm - eff))
        cols[rows] = np.stack((before, after, eff, dur, avg, bmax, lmax, bmin, lmin, resid, dev_, np.zeros(rows.size)), axis=1)
    return cols, types


class RaggedColumn:
    """A list column of events.csv (one vector of `lengths[i]` values per event) as a padded 2-D array: indexing and
    iteration give the per-event vectors; `strings()` gives the ';'-joined `%.16g` text column by column."""

    def __init__(self, data: np.ndarray, lengths: np.ndarray):
        self.data, self.lengths = np.asarray(data, np.float64), np.asarray(lengths, np.int64)

    def __len__(self) -> int:
        return int(self.lengths.size)

    def __getitem__(self, i):
        if isinstance(i, (int, np.integer)):
            return self.data[i, :self.lengths[i]].copy()
        return RaggedColumn(self.data[i], self.lengths[i])

    def __iter__(self):
        return (self.data[i, :self.lengths[i]] for i in range(len(self)))

    def strings(self) -> np.ndarray:
        out = np.full(len(self), "", dtype=object)
        for k in range(self.data.shape[1] if len(self) else 0):      # mosaicConverter.py:139-148 ('%.16g;' joined, last ';' cut)
            sel = self.lengths > k
            if not sel.any():
                break
            txt = np.char.mod("%.16g", self.data[sel, k]).astype(object)
            out[sel] = txt if k == 0 else out[sel] + ";" + txt
        return out


@dataclass
class EventTable:
    """Column-oriented event table (numpy).  `rate` holds every detected event, `events`
    the accepted ones (types 0 and 1) with the full column set; list columns are object arrays of
    float64 vectors until they are serialised."""
    events: dict
    rate: dict

    def __len__(self) -> int:
        return len(self.events["id"])


def build_event_table(*, starts, ends, types, n_levels, edges, level_mean, level_std, overflow, xmin, xmax,
                      samplerate: float, threshold: float, baseline_mean, baseline_std, baseline_block: int,
                      padding: int, first_id: int = 0, time_offset_s: float = 0.0, index_offset: int = 0,
                      block_offset: int = 0, intra_count=None, intra_pairs=None, columns=None,
                      stepfit_params=None) -> EventTable:
    """Per-event columns from the detector / CUSUM+ / step-fit tables (numpy arrays, one row per detected
    event).  `index_offset` is the global sample index of the shard's first owned sample,
    `first_id` the global id of its first event (multi-GPU: pipeline.AnalysisResult).
    `stepfit_params` [E, 6] (stepfit.StepFitTable.params) gives the rc columns of type-1 rows."""
    starts = np.asarray(starts, np.int64); ends = np.asarray(ends, np.int64)
    E = starts.size
    types = np.asarray(types, np.int32).copy()
    nl = np.asarray(n_levels, np.int64)
    edges = np.asarray(edges, np.int64).reshape(E, -1)
    mu = np.asarray(level_mean, np.float64).reshape(E, -1)
    sd = np.asarray(level_std, np.float64).reshape(E, -1)
    ML = mu.shape[1] if E else 0
    fs = float(samplerate)
    if columns is None:
        cols, types = event_columns_host(types, nl, edges, mu, sd, overflow, xmin, xmax)
    else:
        cols, types = np.asarray(columns[0], np.float64).reshape(E, 12), np.asarray(columns[1], np.int32).copy()
    ids = first_id + np.arange(E, dtype=np.int64)
    t_start = time_offset_s + (index_offset + starts) / fs
    t_end = time_offset_s + (index_offset + ends) / fs
    # `block_offset`: samples the baseline table starts before the first owned sample (a shard's left halo)
    blk = np.minimum((starts + int(block_offset)) // int(baseline_block), len(baseline_mean) - 1) if E else np.zeros(0, np.int64)
    # intra-event crossings: ';'-joined start;end;start;end... in us on the event file's time axis (0 = window start)
    crossing_txt = np.array([""] * E, dtype=object)
    ic = np.zeros(E, np.int64)
    if intra_count is not None and E:
        ic = np.asarray(intra_count, np.int64)
        ip = np.asarray(intra_pairs, np.int64).reshape(E, -1)
        kmax = ip.shape[1] // 2
        crossing_txt = RaggedColumn(ip * (1e6 / fs), 2 * np.minimum(ic, kmax)).strings()
    rate = {"id": ids, "type": types, "start_time_s": t_start, "end_time_s": t_end,
            "intra_crossing_times_us": crossing_txt,
            "local_stdev": np.asarray(baseline_std, np.float64)[blk] if E else np.zeros(0),
            "local_baseline": np.asarray(baseline_mean, np.float64)[blk] if E else np.zeros(0)}

    ok = np.nonzero(np.isin(types, GOOD_TYPES))[0]
    n = ok.size
    rc1, rc2 = np.zeros(n), np.zeros(n)
    if stepfit_params is not None and n:
        sp = np.asarray(stepfit_params, np.float64).reshape(E, 6)[ok]
        fitted = types[ok] == TYPE_STEPFIT
        rc1 = np.where(fitted, sp[:, 4] * (1e6 / fs), 0.0)
        rc2 = np.where(fitted, sp[:, 5] * (1e6 / fs), 0.0)
    L = nl[ok]
    col = np.arange(ML)[None, :]
    valid = col < L[:, None]                       # levels of the window
    length = np.where(valid, edges[ok, 1:ML + 1] - edges[ok, :ML], 0).astype(np.float64)
    m = np.where(valid, mu[ok], 0.0)
    s = np.where(valid, sd[ok], 0.0)
    c = cols[ok]
    before, after, eff, dur_in, avg_block = c[:, 0], c[:, 1], c[:, 2], c[:, 3], c[:, 4]
    sgn = np.where(eff >= 0, 1.0, -1.0)
    block = sgn[:, None] * (eff[:, None] - m)      # blockage of every level; the first / last entries are the baselines
    rows = np.arange(n)
    if n:
        block[rows, 0] = before - eff              # mosaicConverter.py:131-132
        block[rows, np.maximum(L - 1, 0)] = after - eff
    us = 1e6 / fs
    with np.errstate(invalid="ignore", divide="ignore"):
        aeff = np.abs(eff)
        lists = {"level_current_pA": RaggedColumn(m, L), "level_duration_us": RaggedColumn(length * us, L),
                 "blockages_pA": RaggedColumn(np.where(valid, block, 0.0), L), "stdev_pA": RaggedColumn(s, L)}
        ts = t_start[ok]
        delay = np.empty(n)
        if n:
            delay[0] = ts[0]
            delay[1:] = ts[1:] - ts[:-1]                                   # mosaicConverter.py:73-76
        events = {"id": ids[ok], "type": types[ok].astype(np.int64), "start_time_s": ts, "event_delay_s": delay,
                  "duration_us": (ends[ok] - starts[ok]) * us, "threshold": np.full(n, float(threshold)),
                  "baseline_before_pA": before, "baseline_after_pA": after, "effective_baseline_pA": eff,
                  "area_pC": avg_block * dur_in / fs, "average_blockage_pA": avg_block,
                  "relative_average_blockage": avg_block / aeff, "max_blockage_pA": c[:, 5],
                  "relative_max_blockage": c[:, 5] / aeff, "max_blockage_duration_us": c[:, 6] * us,
                  "n_levels": L - 1, "intra_crossings": ic[ok], "rc_const1_us": rc1,
                  "rc_const2_us": rc2, "residual_pA": c[:, 9], "max_deviation_pA": c[:, 10],
                  "min_blockage_pA": c[:, 7], "relative_min_blockage": c[:, 7] / aeff,
                  "min_blockage_duration_us": c[:, 8] * us, **lists}
    return EventTable(events=events, rate=rate)


def _table_from_host(tabs: dict, levels, types, y, win_start, win_end, baseline, **kw) -> EventTable:
    """`build_event_table` over the host columns of an analyzer (pipeline.AnalysisResult.columns), with the derived
    columns and the extrema of the windows y[win_start:win_end] computed on the device (`event_columns`)."""
    lo, hi = event_extrema(y, win_start, win_end)
    cols, ty = event_columns(levels, types, lo, hi)
    return build_event_table(columns=(cols.cpu().numpy(), ty.cpu().numpy()), starts=tabs["starts"], ends=tabs["ends"],
                             types=tabs["types"], n_levels=tabs["n_levels"], edges=tabs["edges"], level_mean=tabs["mean"],
                             level_std=tabs["std"], overflow=tabs["overflow"], xmin=lo.cpu().numpy(), xmax=hi.cpu().numpy(),
                             baseline_mean=baseline.mean, baseline_std=baseline.std, intra_count=tabs.get("intra_count"),
                             intra_pairs=tabs.get("intra_pairs"), stepfit_params=tabs.get("stepfit_params"), **kw)


def event_table_from_result(an, r, *, samplerate: float, time_offset_s: float = 0.0, index_offset: int = 0) -> EventTable:
    """Event table of one `pipeline.TraceAnalyzer.run` result (device -> host, then
    `build_event_table`)."""
    return _table_from_host(an.tables_to_host(r), r.levels, r.types, r.detect_trace, r.win_start, r.win_end, r.baseline,
                            samplerate=samplerate, threshold=an.threshold, baseline_block=an.block,
                            padding=an.event_padding, first_id=r.first_event_id, time_offset_s=time_offset_s,
                            index_offset=index_offset, block_offset=r.lo_halo)


def event_table_from_stream(san, rs, *, samplerate: float, time_offset_s: float = 0.0, index_offset: int = 0) -> EventTable:
    """Event table of one `pipeline.StreamingAnalyzer.run_from_host` result: the tables are already on
    the host; only the per-event extrema are taken from the device-resident filtered trace (windows =
    event +- event_padding, clipped to the rank's owned samples)."""
    t = rs.tables
    pad, n = int(san.kw.get("event_padding", 100)), int(rs.filtered.numel())
    dev = rs.filtered.device
    w0 = torch.from_numpy(np.clip(t["starts"] - pad, 0, n)).to(dev)
    w1 = torch.from_numpy(np.clip(t["ends"] + pad, 0, n)).to(dev)
    # the level rows went to the host sub-shard by sub-shard: one upload for the derived columns
    types = torch.from_numpy(np.ascontiguousarray(t["types"])).to(dev)
    return _table_from_host(t, cusum.LevelTable.from_columns(t, dev), types, rs.filtered, w0, w1, rs.baseline,
                            samplerate=samplerate, threshold=float(san.kw.get("threshold", 5.0)), baseline_block=san.block,
                            padding=pad, first_id=rs.first_event_id, time_offset_s=time_offset_s, index_offset=index_offset)


def _write_csv(path: str, columns, table: dict) -> None:
    import pandas as pd
    df = pd.DataFrame({c: (np.zeros(len(table[c])) if isinstance(table[c], RaggedColumn) else table[c]) for c in columns}, columns=columns)
    for c in columns:
        if isinstance(table[c], RaggedColumn):
            df[c] = table[c].strings()
    df.to_csv(path, index=False, encoding="utf-8")


def write_analysis_dir(path: str, table: EventTable, *, baseline_mean, baseline_std, baseline_block: int,
                       samplerate: float, threshold: float, hysteresis: float, cutoff: float, poles: int,
                       extra_summary: dict | None = None, event_samples=None, time_offset_s: float = 0.0,
                       append: bool = False, intra_threshold: float = 0.0, intra_hysteresis: float = 0.0,
                       stepfit_samples: int = 0, stepfit_fallback: bool = False) -> None:
    """Write `events.csv`, `rate.csv`, `baseline.csv`, `summary.txt` and (if `event_samples`
    is given) `events/event_%08d.csv` under `path`.

    `event_samples` maps event id -> (window_start_index, samples float array, edges, level
    means[, step-fit parameters]): the rows of the per-event file are `time_us, current_pA, cusum_fit`
    (`readevents.py:1334-1337` names them time, current, cusum) WITH a header line, because
    the consumer reads them with an implicit header row (`readevents.py:1319`).  An entry with
    parameters (a type-1 event) gets a fourth column `stepfit`, the fitted step response f(t).
    `stepfit_samples` > 0 (the analyzer's length threshold of the fit) and `stepfit_fallback` (the analyzer fitted
    the events CUSUM+ left without a sub-level) are recorded in summary.txt."""
    os.makedirs(os.path.join(path, "events"), exist_ok=True)
    _write_csv(os.path.join(path, "events.csv"), EVENT_COLUMNS, table.events)
    _write_csv(os.path.join(path, "rate.csv"), RATE_COLUMNS, table.rate)
    fs = float(samplerate)
    nb = len(baseline_mean)
    _write_csv(os.path.join(path, "baseline.csv"), ["time_s", "baseline_pA", "stdev_pA"],
               {"time_s": time_offset_s + np.arange(nb) * (int(baseline_block) / fs),
                "baseline_pA": np.asarray(baseline_mean, np.float64), "stdev_pA": np.asarray(baseline_std, np.float64)})
    # summary.txt: consumers parse by SUBSTRING (plot-trace.py:190-203, readevents.py:73-79), so no
    # other key may contain 'threshold', 'hysteresis', 'cutoff' or 'poles'
    summary = {"threshold": repr(float(threshold)), "hysteresis": repr(float(hysteresis)), "cutoff": str(int(cutoff)),
               "poles": str(int(poles)), "intra_threshold": repr(float(intra_threshold)) if intra_threshold else "0",
               "intra_hysteresis": repr(float(intra_hysteresis)) if intra_hysteresis else "0", "samplerate": repr(fs),
               "baseline_block_samples": str(int(baseline_block)), "events_detected": str(len(table.rate["id"])),
               "events_accepted": str(len(table))}
    if stepfit_samples:
        summary["stepfit_samples"] = str(int(stepfit_samples))
    if stepfit_fallback:
        summary["stepfit_fallback"] = "1"
    for k, v in (extra_summary or {}).items():
        if any(w in k for w in ("threshold", "hysteresis", "cutoff", "poles")):
            raise ValueError(f"summary key {k!r} would be mis-parsed by the consumers' substring match")
        summary[k] = str(v)
    # the two intra_ keys go last and the plain keys first: plot-trace.py skips lines containing 'intra'
    with open(os.path.join(path, "summary.txt"), "w") as f:
        for k, v in summary.items():
            f.write(f"{k}={v}\n")
    if event_samples:
        us = 1e6 / fs
        from .stepfit import model
        for eid, entry in event_samples.items():
            w0, x, ed, mu = entry[:4]
            params = entry[4] if len(entry) > 4 else None
            x = np.asarray(x, np.float64)
            fit = np.empty_like(x)
            for i in range(len(ed) - 1):
                fit[ed[i]:ed[i + 1]] = mu[i]
            t = np.arange(x.size) * us
            with open(os.path.join(path, "events", "event_%08d.csv" % int(eid)), "w") as f:
                if params is None:
                    f.write("time_us,current_pA,cusum_fit\n")
                    np.savetxt(f, np.c_[t, x, fit], delimiter=",", fmt="%.16g")
                else:
                    f.write("time_us,current_pA,cusum_fit,stepfit\n")
                    np.savetxt(f, np.c_[t, x, fit, model(params, x.size)], delimiter=",", fmt="%.16g")


def gather_event_samples(an, r, ids, table: EventTable) -> dict:
    """Samples + step fit of the chosen event ids (global ids) for the per-event files; type-1 events also
    carry their step-response parameters (the `stepfit` column)."""
    tabs = {k: v for k, v in zip(("w0", "w1"), (r.win_start.cpu().numpy(), r.win_end.cpu().numpy()))}
    nl = r.levels.n_levels.cpu().numpy(); ed = r.levels.edges.cpu().numpy(); mu = r.levels.mean.cpu().numpy()
    sf = getattr(r, "stepfit", None)
    typ = r.types.cpu().numpy() if sf is not None else None
    par = sf.params.cpu().numpy() if sf is not None else None
    out = {}
    for eid in ids:
        i = int(eid) - r.first_event_id
        if i < 0 or i >= len(nl) or nl[i] <= 0:
            continue
        a, b = int(tabs["w0"][i]), int(tabs["w1"][i])
        entry = (a, r.detect_trace[a:b].cpu().numpy(), ed[i, :nl[i] + 1].astype(np.int64), mu[i, :nl[i]])
        if sf is not None and typ[i] == TYPE_STEPFIT:
            entry = entry + (par[i].copy(),)          # u1, u2 are relative to the window start, as the samples
        out[int(eid)] = entry
    return out
