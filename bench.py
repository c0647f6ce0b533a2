#!/usr/bin/env python
"""Benchmark of the raw-trace hot path (BASELINE.json metric, config C2 per GPU).

    python bench.py --gpus N --steps K --warmup W            # ours (one rank per GPU)
    python bench.py --impl reference ...                      # the CPU path on host cores

A step = one pass of the hot path over one synthetic 10-minute Chimera trace per GPU
(2 499 999 600 uint16 samples at 4.17 MHz, 1000 two-level events/s): exact global median
-> fused dequantise + 8-pole 100 kHz Bessel filtfilt -> baseline blocks -> threshold
detection -> CUSUM+ segmentation of every detected event.  `value` is with the raw codes
resident in HBM; `e2e` starts from pinned host memory and ends with the event/level
tables back on the host.  Inputs (5 GB) are far larger than the 126 MB L2, so no explicit
L2 flush is needed between iterations.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

C2_SAMPLES = 2_499_999_600
C5_SAMPLES = 14_999_997_600
CUTOFF, ORDER = 100_000.0, 8
THRESHOLD, HYSTERESIS = 5.0, 1.0
BASELINE_BLOCK = 1 << 20
BASELINE_MIN, BASELINE_MAX = 4700.0, 5300.0
EVENT_PAD, MINPOINTS, MAXPOINTS = 100, 8, 100_000
E2E_SHARDS = 16                      # time sub-shards of the streamed end-to-end run (pipeline.StreamingAnalyzer)
CUSUM_DELTA, CUSUM_H = 400.0, 10.0
# --dump-outputs: 512 windows of 8192 filtered samples (17 MB) and 65 536 event rows (30 MB) at most
DUMP_WINDOWS, DUMP_WINDOW, DUMP_EVENTS, DUMP_SEED = 512, 8192, 1 << 16, 0
DUMP_BUDGET = 64_000_000
METRIC = "Msamples/s filtered+CUSUM-segmented"
FILTER_BYTES_PER_SAMPLE = 6.0     # 2 B uint16 read + 4 B float32 written (SURVEY.md 8d)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (matched by nvidia-smi's own timestamps:
    its stdout reaches a pipe in bursts)."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "10"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    @staticmethod
    def _stamp(txt: str) -> float:
        import datetime
        return datetime.datetime.strptime(txt.strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()

    def summary(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.3)                      # let the tail of the stream arrive
        self.proc.terminate()
        time.sleep(0.1)
        parsed = []
        for line in self.rows:
            p = [x.strip() for x in line.split(",")]
            try:
                parsed.append((self._stamp(p[0]), float(p[1]), float(p[2]), p[4:8]))
            except Exception:
                continue
        inside = [r for r in parsed if t0 - 0.005 <= r[0] <= t1 + 0.03]
        note = None
        if not inside and parsed:            # a very short region: the samples nearest to it
            mid = 0.5 * (t0 + t1)
            inside = sorted(parsed, key=lambda r: abs(r[0] - mid))[:3]
            note = "no sample fell inside the timed region; nearest samples used"
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no nvidia-smi sample"]}
        reasons = set()
        for _, _, _, flags in inside:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), flags):
                if v.lower().startswith("active"):
                    reasons.add(name)
        out = {"sm_mhz": float(np.median([r[1] for r in inside])), "sm_max_mhz": float(max(r[2] for r in inside)),
               "reasons": sorted(reasons), "samples": len(inside)}
        if note:
            out["note"] = note
        return out


# ------------------------------------------------------------------------ CPU baseline
def _cpu_chunk(args):
    """The reference's call sequence on one chunk (oracle = port of it; the arithmetic is
    the same scipy/numpy routines the reference calls)."""
    seed, n = args
    from cusumtools_b200 import synth
    from oracle import c_twin, events_oracle as eo, trace_oracle as to
    codes, _ = synth.c1_trace(n=n, n_events=(n - 4000) // synth.EVENT_PERIOD, seed=seed)
    t0 = time.perf_counter()
    data = to.scale_raw_data(codes, synth.CHIMERA_SETTINGS)                  # plot-trace.py:272-287
    y = to.filter_data(data, synth.FS, CUTOFF, ORDER).astype(np.float32)     # plot-trace.py:313-320
    blk = 1 << 16
    c0 = np.float32(0.5 * (BASELINE_MIN + BASELINE_MAX))
    sh = eo.stats_shift(300.0, blk)
    mean, std = eo.baseline_from_stats(*c_twin.block_stats(y, blk, BASELINE_MIN, BASELINE_MAX, c0, sh), c0, sh)
    s, e, _ = c_twin.detect_events(y, blk, *eo.thresholds(mean, std, THRESHOLD, HYSTERESIS))
    w0, w1, typ = eo.event_windows(s, e, n, EVENT_PAD, MINPOINTS, MAXPOINTS)
    ok = typ == 0
    offs = np.concatenate(([0], np.cumsum((w1 - w0)[ok])))
    flat = np.concatenate([y[a:b] for a, b in zip(w0[ok], w1[ok])]) if ok.any() else np.zeros(0, np.float32)
    c_twin.cusum_batch(flat, offs, CUSUM_DELTA, CUSUM_H)
    return time.perf_counter() - t0, n, int(ok.sum())


def cpu_baseline_single(n=1 << 24):
    """1 process / 1 thread, as the reference runs (single-threaded Tk script)."""
    best = None
    for r in range(2):
        dt, nn, ne = _cpu_chunk((r, n))
        best = dt if best is None else min(best, dt)
    return {"value": n / best / 1e6, "unit": "Msamples/s", "cores": 1, "kind": "port",
            "sample": f"{n} samples ({n / 4166666.0:.1f} s of the same synthetic trace), best of 2; "
                      "scale_raw_data + np.pad(median)+filtfilt (scipy) + detection + CUSUM (C twin of the oracle)"}


def run_reference(args):
    """--impl reference: the CPU path on all host cores (chunks of the same workload, one
    process per core, each chunk median-padded on its own — a throughput baseline)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = len(os.sched_getaffinity(0))
    n_chunk = 1 << 23
    times = []
    with mp.get_context("fork").Pool(cores) as pool:
        for it in range(args.warmup + args.steps):
            res = pool.map(_cpu_chunk, [(it * cores + c, n_chunk) for c in range(cores)])
            # all chunks run concurrently; the step takes as long as the slowest one
            # (synthetic-trace generation inside the workers is not part of the path)
            if it >= args.warmup:
                times.append(max(r[0] for r in res))
    total = n_chunk * cores
    ms = 1e3 * float(np.mean(times))
    val = total / (ms / 1e3) / 1e6
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "Msamples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "C2: 10-min 4.17 MHz Chimera trace, 8-pole 100 kHz Bessel filtfilt + threshold "
                                   "detection + CUSUM+ (bounded sample per step)", "sample_per_step": total},
            "cpu_baseline": {"value": val, "unit": "Msamples/s", "cores": cores, "kind": "port",
                             "sample": f"{cores} chunks x {n_chunk} samples per step, one process per core; the "
                                       "reference is pure Python over numpy/scipy (nothing to compile into "
                                       "oracle/_ref), so the oracle port of its call sequence is timed"},
            "e2e": {"value": val, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def side_kernels(torch, dev, peak):
    """Kernel-only numbers of the two stages the C2 step does not exercise at their own config shape
    (reported next to the headline, not part of `value`): CUSUM+ on pre-extracted events (C3: 1 M
    events) and the Welch PSD (C4 shape, 2^20-point segments over 2^28 samples); 4 B/sample algorithmic."""
    from cusumtools_b200 import cusum, psd, synth
    out = {}
    x, offs, _ = synth.c3_events_device(1_000_000, dev)
    w0, w1 = offs[:-1].contiguous(), offs[1:].contiguous()
    cusum.cusum_levels(x, w0, w1, delta=CUSUM_DELTA, h=CUSUM_H)
    a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); a.record()
    for _ in range(3):
        cusum.cusum_levels(x, w0, w1, delta=CUSUM_DELTA, h=CUSUM_H)
    b.record(); torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 3
    out["cusum_c3_1M_events"] = {"Msamples_per_s": x.numel() / ms / 1e3, "Mevents_per_s": 1_000_000 / ms / 1e3,
                                   "hbm_frac": 4.0 * x.numel() / ms / 1e6 / peak}
    del x, offs, w0, w1
    g = torch.Generator(device=dev); g.manual_seed(3)
    y = torch.randn(1 << 28, generator=g, device=dev) * 24 + 5000
    psd.welch_sums(y, 1 << 20, shift=5000.0)
    torch.cuda.synchronize(); a.record()
    for _ in range(3):
        psd.welch_sums(y, 1 << 20, shift=5000.0)
    b.record(); torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 3
    out["welch_c4_2p20_segments"] = {"Msamples_per_s": y.numel() / ms / 1e3, "hbm_frac": 4.0 * y.numel() / ms / 1e6 / peak}
    return out


# ------------------------------------------------------------------------- parity at size
def parity_at_size(torch, dist, group, an, raw, r, S, lo_h, n_own, rank, world):
    """Outside the timed region: the CUDA path against the oracle AT THE BENCHMARKED SIZE.  Whole baseline blocks of
    the device trace (one around 1e9 samples, two straddling sample 2^31, the last ones of the trace; at N > 1 also the
    blocks either side of the shard boundaries) are pulled to the host and run through the oracle chain:
    filter (reference call sequence, float64) within 0.05 pA; block sums, baseline rows, detector lines, event indices
    and CUSUM+ levels `array_equal` on the identical float32 input (C twin of oracle/events_oracle.py); the exact median
    against an independent torch.bincount of all codes (summed over ranks)."""
    from cusumtools_b200 import filters
    from oracle import c_twin, events_oracle as eo, trace_oracle as to
    dev = raw.device
    n_ext = raw.numel()
    blk = BASELINE_BLOCK
    mask = filters.chimera_bitmask(S)
    out = {"windows": 0, "samples": 0, "max_abs_pA": 0.0, "blocks_equal": True, "events_equal": True, "levels_equal": True,
           "events_checked": 0, "levels_checked": 0, "beyond_2p31": False}
    # ---- exact median, independently: a plain histogram of the OWNED codes (torch), all ranks summed
    hist = torch.zeros(65536, dtype=torch.int64, device=dev)
    own = raw[lo_h:lo_h + n_own]
    for a in range(0, n_own, 1 << 28):
        hist += torch.bincount((own[a:a + (1 << 28)].to(torch.int32) & mask), minlength=65536)
    if group is not None:
        dist.all_reduce(hist, group=group)
    cdf = torch.cumsum(hist, 0).cpu().numpy()
    ntot = int(cdf[-1])
    med = (int(np.searchsorted(cdf, (ntot - 1) // 2 + 1)), int(np.searchsorted(cdf, ntot // 2 + 1)))
    out["median_exact"] = bool(tuple(r.median_codes) == med)
    pad_value = float(np.median(to.scale_raw_data(np.array(med, dtype=np.uint16), S)))
    out["pad_value_equal"] = bool(pad_value == r.pad_value)
    # ---- windows of whole blocks, in extended-trace coordinates
    nb = -(-n_ext // blk)
    wins = []
    def add(b0, b1):
        b0, b1 = max(0, b0), min(nb, b1)
        if b1 > b0 and (b0, b1) not in wins:
            wins.append((b0, b1))
    add(min(nb - 1, 1_000_000_000 // blk), min(nb - 1, 1_000_000_000 // blk) + 1)
    if n_ext > (1 << 31) + blk:
        add((1 << 31) // blk - 1, (1 << 31) // blk + 1)
        out["beyond_2p31"] = True
    add(nb - 2, nb)
    if lo_h:
        add(lo_h // blk - 1, lo_h // blk + 1)
    if n_ext - lo_h - n_own:
        add((lo_h + n_own) // blk - 1, (lo_h + n_own) // blk + 1)
    y_all = r.detect_trace
    starts = (r.events.starts + lo_h).cpu().numpy()
    ends = (r.events.ends + lo_h).cpu().numpy()
    w0s, w1s, typ = r.win_start.cpu().numpy(), r.win_end.cpu().numpy(), r.types.cpu().numpy()
    bl = r.baseline
    sign, ts, te = bl.sign, bl.t_start, bl.t_end
    cnt_g, s1_g, s2_g = (bl.dev[k].cpu().numpy() for k in ("cnt", "s1", "s2"))
    margin = 8192
    alpha_design = None
    for (b0, b1) in wins:
        p0, p1 = b0 * blk, min(b1 * blk, n_ext)
        q0, q1 = max(0, p0 - margin), min(n_ext, p1 + margin)
        codes = raw[q0:q1].cpu().numpy()
        x = to.scale_raw_data(codes, S)
        # the reference call sequence (plot-trace.py:313-320) on the neighbourhood; at a true end of the trace the pad is
        # the GLOBAL median, elsewhere the margin keeps the window's own pad out of reach
        from scipy.signal import bessel, filtfilt
        b_, a_ = bessel(ORDER, 2.0 * CUTOFF / np.floor(np.squeeze(S["ADCSAMPLERATE"])), "low")
        padded = np.pad(x, 1000, mode="constant", constant_values=pad_value)
        y_ref = filtfilt(b_, a_, padded, padtype=None)[1000:-1000]
        lo_ok = 0 if (q0 == 0 and lo_h == 0 and rank == 0) else p0 - q0
        hi_ok = (q1 - q0) if (q1 == n_ext and n_ext - lo_h - n_own == 0 and rank == world - 1) else p1 - q0
        if q0 == 0 and not (lo_h == 0 and rank == 0):
            lo_ok = max(lo_ok, margin)
        if q1 == n_ext and not (n_ext - lo_h - n_own == 0 and rank == world - 1):
            hi_ok = min(hi_ok, q1 - q0 - margin)
        y_gpu = y_all[q0:q1].cpu().numpy()
        err = float(np.abs(y_gpu[lo_ok:hi_ok].astype(np.float64) - y_ref[lo_ok:hi_ok]).max()) if hi_ok > lo_ok else 0.0
        out["max_abs_pA"] = max(out["max_abs_pA"], err)
        out["windows"] += 1
        out["samples"] += int(p1 - p0)
        # ---- stage 2 on the identical float32 input
        yw = np.ascontiguousarray(y_all[p0:p1].cpu().numpy())
        c0 = np.float32(bl.dev["c0"])
        sh = int(bl.dev["shift"])
        cnt, s1, s2 = c_twin.block_stats(yw, blk, BASELINE_MIN, BASELINE_MAX, c0, sh)
        ok = (np.array_equal(cnt, cnt_g[b0:b1]) and np.array_equal(s1, s1_g[b0:b1]) and np.array_equal(s2, s2_g[b0:b1]))
        valid = cnt >= 16
        if valid.all():
            mean, std = eo.baseline_from_stats(cnt, s1, s2, c0, sh)
            sg, t_s, t_e = eo.thresholds(mean, std, THRESHOLD, HYSTERESIS)
            ok = ok and np.array_equal(mean, bl.mean[b0:b1]) and np.array_equal(std, bl.std[b0:b1])
            ok = ok and np.array_equal(sg, sign[b0:b1]) and np.array_equal(t_s, ts[b0:b1]) and np.array_equal(t_e, te[b0:b1])
        out["blocks_equal"] = bool(out["blocks_equal"] and ok)
        # ---- detection: the oracle's state machine over the window with the device's lines; the state at the window
        # start comes from the device's own event list (an event that straddles p0)
        inside0 = bool(np.any((starts < p0) & (ends >= p0)))
        s_o, e_o, _ = c_twin.detect_events(yw, blk, sign[b0:b1], ts[b0:b1], te[b0:b1], state_in=inside0)
        s_o, e_o = s_o + p0, e_o + p0
        own_lo, own_hi = lo_h, lo_h + n_own
        keep_o = (s_o >= own_lo) & (s_o < own_hi)
        sel = (starts >= p0) & (starts < p1) & (ends < p1)
        ev_ok = np.array_equal(starts[sel], s_o[keep_o]) and np.array_equal(ends[sel], e_o[keep_o])
        out["events_equal"] = bool(out["events_equal"] and ev_ok)
        out["events_checked"] += int(sel.sum())
        # ---- CUSUM+ of the accepted events whose window lies inside [p0, p1)
        if r.levels is not None:
            pick = np.nonzero(sel & (typ == 0) & (w0s >= p0) & (w1s <= p1))[0]
            if pick.size:
                offs = np.concatenate(([0], np.cumsum((w1s - w0s)[pick])))
                flat = np.concatenate([yw[a - p0:b - p0] for a, b in zip(w0s[pick], w1s[pick])])
                nl, ed, mu, sd, ov = c_twin.cusum_batch(flat, offs, CUSUM_DELTA, CUSUM_H, r.levels.max_levels)
                idx = torch.from_numpy(pick).to(dev)
                g_nl = r.levels.n_levels[idx].cpu().numpy(); g_ed = r.levels.edges[idx].cpu().numpy()
                g_mu = r.levels.mean[idx].cpu().numpy(); g_sd = r.levels.std[idx].cpu().numpy()
                lv_ok = np.array_equal(g_nl, nl) and np.array_equal(g_ed, ed)
                rows = np.arange(mu.shape[1])[None, :] < nl[:, None]
                lv_ok = lv_ok and np.array_equal(g_mu[rows], mu[rows]) and np.array_equal(g_sd[rows], sd[rows])
                out["levels_equal"] = bool(out["levels_equal"] and lv_ok)
                out["levels_checked"] += int(nl.sum())
    flags = torch.tensor([int(out["blocks_equal"]), int(out["events_equal"]), int(out["levels_equal"]), int(out["median_exact"]),
                          int(out["pad_value_equal"])], dtype=torch.int64, device=dev)
    worst = torch.tensor([out["max_abs_pA"]], dtype=torch.float64, device=dev)
    tot = torch.tensor([out["windows"], out["samples"], out["events_checked"], out["levels_checked"]], dtype=torch.int64, device=dev)
    if group is not None:
        dist.all_reduce(flags, op=dist.ReduceOp.MIN, group=group)
        dist.all_reduce(worst, op=dist.ReduceOp.MAX, group=group)
        dist.all_reduce(tot, group=group)
    f = flags.cpu().numpy(); t = tot.cpu().numpy()
    out.update(blocks_equal=bool(f[0]), events_equal=bool(f[1]), levels_equal=bool(f[2]), median_exact=bool(f[3]),
               pad_value_equal=bool(f[4]), max_abs_pA=float(worst.item()), windows=int(t[0]), samples=int(t[1]),
               events_checked=int(t[2]), levels_checked=int(t[3]), tolerance_pA=0.05,
               note="whole baseline blocks of the benchmarked device trace against the oracle chain; filter vs the reference's "
                    "float64 call sequence, stages 2-3 array_equal on identical float32 input; all ranks (flags AND, error MAX)")
    return out


def dump_outputs(path, r, extra=None):
    """Writes what one step of the timed path returned (the AnalysisResult of TraceAnalyzer.run) as float64 .npy files,
    float32 for the filtered trace, so that two builds can be compared output for output.  The filtered trace is sampled
    in DUMP_WINDOWS contiguous windows and the event rows in DUMP_EVENTS rows, both at positions fixed by DUMP_SEED;
    `*_index` files say which.  level_mean / level_std hold each sampled event's first level_count entries, event after
    event: the table's entries beyond an event's level count are never written by the kernel."""
    import torch
    f64 = lambda t: t.cpu().numpy().astype(np.float64)
    out = {}
    y = r.filtered
    n = y.numel()
    if n <= DUMP_WINDOWS * DUMP_WINDOW:
        starts, w = np.zeros(1, np.int64), n
    else:
        stride = n // DUMP_WINDOWS
        rng = np.random.default_rng(DUMP_SEED)
        starts = np.arange(DUMP_WINDOWS, dtype=np.int64) * stride + rng.integers(0, stride - DUMP_WINDOW + 1, DUMP_WINDOWS)
        w = DUMP_WINDOW
    idx = torch.from_numpy(starts).to(y.device)[:, None] + torch.arange(w, device=y.device)
    out["filtered"] = y[idx].cpu().numpy()
    out["filtered_index"] = starts.astype(np.float64)
    n_ev = r.events.starts.numel()
    rows = np.arange(n_ev)
    if n_ev > DUMP_EVENTS:
        rows = np.sort(np.random.default_rng(DUMP_SEED).choice(n_ev, DUMP_EVENTS, replace=False))
    sel = torch.from_numpy(rows).to(y.device)
    out["event_index"] = rows.astype(np.float64)
    out["event_start"], out["event_end"] = f64(r.events.starts[sel]), f64(r.events.ends[sel])
    out["window_start"], out["window_end"], out["event_type"] = f64(r.win_start[sel]), f64(r.win_end[sel]), f64(r.types[sel])
    if r.levels is not None:
        lv = r.levels
        nl = f64(lv.n_levels[sel])
        fit = np.arange(lv.max_levels)[None, :] < nl[:, None]
        out["level_count"], out["level_edges"], out["level_overflow"] = nl, f64(lv.edges[sel]), f64(lv.overflow[sel])
        out["level_mean"], out["level_std"] = f64(lv.mean[sel])[fit], f64(lv.std[sel])[fit]
    bl = r.baseline
    for k in ("mean", "std", "sign", "t_start", "t_end"):
        out["baseline_" + k] = np.asarray(getattr(bl, k), dtype=np.float64)
    out["pad_value"] = np.array([r.pad_value])
    out["median_codes"] = np.array(r.median_codes, dtype=np.float64)
    out["event_count"] = np.array([n_ev, r.events.open_start, r.first_event_id, r.total_events], dtype=np.float64)
    out.update(extra or {})
    size = sum(a.nbytes for a in out.values())
    if size > DUMP_BUDGET:
        raise SystemExit(f"--dump-outputs: {size} bytes exceed the {DUMP_BUDGET}-byte budget")
    os.makedirs(path, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(path, k + ".npy"), a)


# ------------------------------------------------------------------------------- ours
def run_ours(args):
    import torch
    import torch.distributed as dist
    from cusumtools_b200 import _lib, cusum, detect, filters, loader, pipeline, psd, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    group = None
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")    # stdout carries exactly one JSON line
        dist.init_process_group("nccl", device_id=dev)
        group = dist.group.WORLD
    S = synth.CHIMERA_SETTINGS
    c5 = args.config == "C5"
    if c5:
        if world < 2:
            raise SystemExit("--config C5 is the 1-hour trace time-sharded over the GPUs of the box: run it with --gpus 2..8")
        lo, hi = pipeline.shard_bounds(C5_SAMPLES, world, rank, BASELINE_BLOCK)
        n_own, total = hi - lo, C5_SAMPLES
        first_index = lo
    else:
        n_own = int(args.samples)
        n_own = n_own // BASELINE_BLOCK * BASELINE_BLOCK if world > 1 else n_own
        total = n_own * world
        first_index = rank * n_own
    halo = pipeline.required_halo(CUTOFF, ORDER, synth.FS, max_event=MAXPOINTS + 2 * EVENT_PAD, block=BASELINE_BLOCK) if world > 1 else 0
    lo_h = halo if rank > 0 else 0
    hi_h = halo if rank < world - 1 else 0
    raw = synth.device_trace(n_own + lo_h + hi_h, dev, seed=1234 + rank, start_index=first_index - lo_h)
    stage_ev = []
    stage_names = ("median", "filter", "baseline", "detect", "cusum") + (("psd", "gather") if c5 else ())
    an = pipeline.TraceAnalyzer(raw.numel(), S, CUTOFF, ORDER, lo_halo=lo_h, hi_halo=hi_h, threshold=THRESHOLD,
                                hysteresis=HYSTERESIS, baseline_block=BASELINE_BLOCK, baseline_min=BASELINE_MIN,
                                baseline_max=BASELINE_MAX, event_padding=EVENT_PAD, minpoints=MINPOINTS,
                                maxpoints=MAXPOINTS, cusum_delta=CUSUM_DELTA, cusum_h=CUSUM_H, group=group, device=dev)
    L_PSD = 1 << 20
    last = {}

    def tail(r, hook):
        """C5 only: the rank's share of the Welch segments (the ones that start in its owned range; the right halo
        holds their overlap), one all_reduce of the L/2+1 sums, and the event / level tables gathered to rank 0."""
        x = r.detect_trace[lo_h:lo_h + n_own + (L_PSD // 2 if rank < world - 1 else 0)]
        acc, nseg = psd.welch_sums(x, L_PSD, shift=r.pad_value)
        acc, nseg = psd.reduce_sums(acc, nseg, group)
        hook("psd")
        cols = {"starts": r.events.starts + (first_index), "ends": r.events.ends + (first_index), "types": r.types,
                "n_levels": r.levels.n_levels, "edges": r.levels.edges, "mean": r.levels.mean, "std": r.levels.std}
        g = pipeline.gather_tables(cols, group, dst=0)
        hook("gather")
        last.update(psd_segments=nseg, psd_sums=acc, gathered=None if g is None else int(g["starts"].shape[0]))
        return acc, g

    def step(hook=None):
        """One pass of the hot path through the public API (pipeline.TraceAnalyzer.run)."""
        h = hook or (lambda name: None)
        r = an.run(raw, stage_hook=hook)
        if c5:
            tail(r, h)
        return r

    def staged_step():
        """The same run with a CUDA event after each stage's launches (only for the per-stage
        breakdown; not part of the timed region)."""
        marks = {}

        def hook(name):
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            marks[name] = e

        torch.cuda.synchronize()
        hook("start")
        step(hook)
        torch.cuda.synchronize()
        stage_ev.append([marks[k] for k in ("start",) + stage_names])

    def fence():
        torch.cuda.synchronize()
        if group is not None:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, k):
        fence()
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        a.record()
        r = None
        for _ in range(k):
            r = fn()
        b.record()
        fence()
        wall = (time.perf_counter() - t0) * 1e3
        ms = torch.tensor([a.elapsed_time(b), wall], dtype=torch.float64, device=dev)
        if group is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX, group=group)
        return float(ms[0]), float(ms[1]), r

    sampler = ClockSampler(local) if rank == 0 else None
    for _ in range(args.warmup):
        step()
    _lib.reset_launch_count()
    tm0 = time.time()
    if args.profile_range:
        torch.cuda.profiler.start()
    dev_ms, wall_ms, res = timed(step, args.steps)
    if args.profile_range:
        torch.cuda.profiler.stop()
    tm1 = time.time()
    launches = _lib.launch_count()
    if args.dump_outputs:
        # before anything else runs the analyzer: `res` is a view of its buffers
        extra = {"psd_sums": np.asarray(last["psd_sums"], dtype=np.float64)} if c5 else None
        dump_outputs(os.path.join(args.dump_outputs, f"rank{rank}") if rank else args.dump_outputs, res, extra)
    for _ in range(2):
        staged_step()
    res = step()
    torch.cuda.synchronize()
    n_events = int(res.events.starts.numel())
    ev_all = torch.tensor([n_events], dtype=torch.int64, device=dev)
    if group is not None:
        dist.all_reduce(ev_all, group=group)
    stage_ms = {nm: float(np.mean([m[i].elapsed_time(m[i + 1]) for m in stage_ev])) for i, nm in enumerate(stage_names)}
    ms_per_step = dev_ms / args.steps
    value = total / (ms_per_step / 1e3) / 1e6

    # ---- parity at the benchmarked size (outside the timed region)
    parity = None if args.no_parity else parity_at_size(torch, dist, group, an, raw, res, S, lo_h, n_own, rank, world)

    # ---- the dominant kernel pair alone (forward + backward filter pass, no host round trip in between),
    # timed with CUDA events on the launching stream: the roofline entry
    med = an.last_median

    def time_pair(stats, cutoff=CUTOFF, iters=3):
        for _ in range(2):
            filters.dequant_filtfilt(raw, S, cutoff, ORDER, median_codes=med, out=an.y, workspace=an.filter_ws, stats=stats)
        fa = torch.cuda.Event(enable_timing=True); fb = torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        fa.record()
        for _ in range(iters):
            filters.dequant_filtfilt(raw, S, cutoff, ORDER, median_codes=med, out=an.y, workspace=an.filter_ws, stats=stats)
        fb.record()
        torch.cuda.synchronize()
        return fa.elapsed_time(fb) / iters

    filt_plain_ms = time_pair(None)
    # the pair as the step runs it: the backward pass also tallies the baseline block sums and leaves the chunk extrema
    # (stage_ms["filter"] minus the exact-median count; timed here through the same entry points, sums only)
    fused_stats = bool(getattr(an, "fuse_stats", False))
    filt_ms = filt_plain_ms
    if fused_stats:
        bl_tmp = detect.new_baseline(raw.numel(), BASELINE_BLOCK, BASELINE_MIN, BASELINE_MAX, dev)
        filt_ms = time_pair(detect.stats_args(bl_tmp, origin=0))
    full_rate_ms = time_pair(None, cutoff=900_000.0) if rank == 0 and not c5 else None
    from cusumtools_b200.design import bessel_lowpass
    decim = filters.scratch_decimation(bessel_lowpass(ORDER, 2.0 * CUTOFF / synth.FS), 1000)

    # ---- end to end: pinned host -> device, pipeline, tables -> host, every step
    e2e = None
    from_file = None
    if not c5:
        host = torch.empty(raw.numel(), dtype=torch.uint16, pin_memory=True)
        host.copy_(raw)
        torch.cuda.synchronize()
        d2h = [0]
        san = pipeline.StreamingAnalyzer(raw.numel(), S, CUTOFF, ORDER, lo_halo=lo_h, hi_halo=hi_h, shards=E2E_SHARDS,
                                         threshold=THRESHOLD, hysteresis=HYSTERESIS, baseline_block=BASELINE_BLOCK,
                                         baseline_min=BASELINE_MIN, baseline_max=BASELINE_MAX, event_padding=EVENT_PAD,
                                         minpoints=MINPOINTS, maxpoints=MAXPOINTS, cusum_delta=CUSUM_DELTA, cusum_h=CUSUM_H,
                                         group=group, device=dev)
        e2e_info = {}

        def e2e_step():
            # pinned H2D cut into time sub-shards; each is filtered, detected, segmented and its tables are
            # copied back (pinned D2H) while the next pieces arrive; returns after the last synchronisation
            r = san.run_from_host(host)
            d2h[0] = sum(v.nbytes for v in r.tables.values())
            e2e_info.update(events=int(r.tables["starts"].shape[0]), redone=r.redone)
            return r.tables

        e2e_step()
        k_e2e = max(2, args.steps // 2)
        e_dev_ms, e_wall_ms, _ = timed(e2e_step, k_e2e)
        e_ms = max(e_dev_ms, e_wall_ms) / k_e2e
        e2e = {"value": total / (e_ms / 1e3) / 1e6, "unit": "Msamples/s", "h2d_bytes_per_step": int(raw.numel() * 2 * world),
               "d2h_bytes_per_step": int(d2h[0] * world), "ms_per_step": e_ms,
               "api": f"pipeline.StreamingAnalyzer.run_from_host ({E2E_SHARDS} time sub-shards overlapped with the pinned H2D copy)",
               "events_rank0": e2e_info.get("events"), "redone": e2e_info.get("redone")}
        # ---- from file: the same streamed run with the codes still in a two-file `.log` series (SURVEY.md 8d)
        if world == 1 and not args.no_file:
            import shutil, tempfile
            import scipy.io as sio
            d = tempfile.mkdtemp(prefix="ct_bench_", dir=args.file_dir)
            try:
                hv = host.numpy()
                cut = (raw.numel() * 3 // 5) & ~1
                for stamp, (a_, b_) in (("20240101_000000", (0, cut)), ("20240101_000600", (cut, raw.numel()))):
                    hv[a_:b_].tofile(os.path.join(d, "bench_" + stamp + ".log"))
                    sio.savemat(os.path.join(d, "bench_" + stamp + ".mat"), S)
                series = loader.ChimeraSeries(os.path.join(d, "bench_20240101_000000.log"))
                rd = series.reader(0.0, None if False else (raw.numel() + 0.5) / series.samplerate)
                assert rd.n == raw.numel(), (rd.n, raw.numel())
                f_info = {}

                def file_step():
                    r = san.run_from_file(rd, threads=args.file_threads)
                    f_info.update(events=int(r.tables["starts"].shape[0]))
                    return r.tables

                file_step()
                f_dev, f_wall, _ = timed(file_step, 2)
                f_ms = max(f_dev, f_wall) / 2
                from_file = {"value": total / (f_ms / 1e3) / 1e6, "unit": "Msamples/s", "ms_per_step": f_ms,
                             "bytes_read_per_step": int(raw.numel() * 2), "files": 2, "reader_threads": args.file_threads,
                             "events": f_info.get("events"),
                             "api": "loader.ChimeraSeries.reader + pipeline.StreamingAnalyzer.run_from_file (preadv into rotating "
                                    "pinned slabs on a worker thread, overlapped with H2D and kernels)",
                             "note": "files written just before the run: reads are served from the page cache"}
                rd.close()
            finally:
                shutil.rmtree(d, ignore_errors=True)

    clocks = sampler.summary(tm0, tm1) if sampler else None
    if rank != 0:
        if group is not None:
            dist.destroy_process_group()
        return
    peak, peak_kind = peaks()
    ach = FILTER_BYTES_PER_SAMPLE * raw.numel() / (filt_ms / 1e3) / 1e9
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
            traffic = tj.get("filter_dram_bytes_per_sample")
            traffic = None if traffic is None else traffic * raw.numel()
            traffic_src = tj.get("source")
    except Exception:
        pass
    workload = ("C5: 1-hour 4.17 MHz Chimera uint16 trace (14 999 997 600 samples) time-sharded over the GPUs with IIR/event halos: "
                "exact global median + 8-pole 100 kHz Bessel filtfilt + baseline + detection + CUSUM+ + Welch PSD (2^20-point "
                "segments, one all_reduce) + event/level tables gathered to rank 0" if c5 else
                "C2: 10-min 4.17 MHz Chimera uint16 trace per GPU, exact median pad + 8-pole 100 kHz "
                "Bessel filtfilt + baseline blocks + threshold detection + CUSUM+ on every detected event")
    line = {
        "metric": METRIC, "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if c5 else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload,
                   "samples_per_gpu": n_own, "halo_samples": halo, "events_per_step": int(ev_all.item()),
                   "l2": "inputs (GBs per GPU) far larger than the 126 MB L2; no flush needed", "parallelism": f"time-sharded x{world}"},
        "events_per_s": int(ev_all.item()) / (ms_per_step / 1e3),
        "wall_ms_per_step": wall_ms / args.steps,
        "stage_ms": stage_ms,
        "parity": parity,
        "roofline": {"kernel": "ct_filter_fwd_kernel + ct_filter_bwd_kernel (fused dequantise + median pad + zero-phase "
                               "Bessel as two TMA-staged lane-sequential passes" + (", baseline block sums tallied in the backward "
                               "pass's epilogue" if fused_stats else "") + "; timed alone, 3 back-to-back calls)", "bound": "hbm",
                     "achieved": ach, "peak": peak, "peak_kind": peak_kind, "unit": "GB/s", "frac": ach / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "kernel_ms": filt_ms,
                     "frac_of_nominal_8000_GBps": ach / 8000.0,      # SURVEY.md 8(d): also against the nominal HBM3e figure
                     "algorithmic_bytes_per_sample": FILTER_BYTES_PER_SAMPLE,
                     "share_of_step": filt_ms / ms_per_step,
                     "scratch_decimation": decim,
                     "filter_only": {"kernel_ms": filt_plain_ms, "frac": FILTER_BYTES_PER_SAMPLE * raw.numel() / (filt_plain_ms / 1e3) / 1e9 / peak,
                                     "note": "the same pair without the fused block sums"},
                     "full_rate_branch": None if full_rate_ms is None else {
                         "cutoff_hz": 900000.0, "kernel_ms": full_rate_ms,
                         "frac": FILTER_BYTES_PER_SAMPLE * raw.numel() / (full_rate_ms / 1e3) / 1e9 / peak,
                         "note": "the reference GUI's default cutoff (plot-trace.py:100-127): the cascade's stop band does not allow "
                                 "a decimated scratch, the forward output crosses HBM at full rate (14 B/sample of traffic)"},
                     "note": "traffic = ncu dram bytes per launch pair at this size (profiles/traffic.json, a constant from the "
                             "committed capture, not re-measured in this run): the forward output crosses HBM once at 1/D rate"},
        "gpu_launches": int(launches),
        "clocks": clocks,
    }
    if e2e is not None:
        line["e2e"] = e2e
    if from_file is not None:
        line["from_file"] = from_file
    if c5:
        line["c5"] = {"total_samples": total, "psd_segments": last.get("psd_segments"), "rows_gathered_on_rank0": last.get("gathered")}
        line["e2e"] = {"value": value, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                       "note": "C5 is generated on the device per rank (30 GB of codes do not fit the bench's host budget); "
                               "the end-to-end figure is measured on C2 (default config)"}
    if world == 1 and not c5:
        line["other_kernels"] = side_kernels(torch, dev, peak)
    if world == 1 and not args.no_cpu:
        line["cpu_baseline"] = cpu_baseline_single()
    emit(line)
    if group is not None:
        dist.destroy_process_group()


_RESULT_FD = None


def emit(line: dict) -> None:
    """The one JSON line, written to the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


def main():
    # stdout must carry exactly one JSON line: libraries that write to file descriptor 1 (NCCL prints its
    # version banner there) are sent to stderr for the whole run, the result goes to the saved descriptor
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--samples", type=int, default=C2_SAMPLES, help="samples per GPU (default: config C2)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--config", default="C2", choices=["C2", "C5"],
                    help="C2: 10-min trace per GPU (weak scaling, the default); C5: the 1-hour trace time-sharded over --gpus ranks, "
                         "with the Welch PSD reduce and the table gather inside the step")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle comparison at the benchmarked size")
    ap.add_argument("--no-file", action="store_true", help="skip the from-file leg (writes the trace to --file-dir first)")
    ap.add_argument("--file-dir", default=None, help="directory for the from-file leg's temporary .log series (default: the system temp dir)")
    ap.add_argument("--file-threads", type=int, default=max(1, min(16, os.cpu_count() or 8)),
                    help="reader threads of the from-file leg (default: the host cores, at most 16: 17.4 against 15.8 Gsamples/s with 8)")
    ap.add_argument("--profile-range", action="store_true",
                    help="bracket the timed region with cudaProfilerStart/Stop (ncu --profile-from-start off)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (sampled to at most 64 MB; rank r > 0 "
                         "of a multi-GPU run under DIR/rank<r>)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
