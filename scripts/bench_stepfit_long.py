"""Long-window step-response fit (ct_stepfit_long_batch) timings on one GPU, in one run:
  * step_fit_long's kernel alone on --events windows (synth.short_events_device: pulses of 8 000-100 000 samples,
    log-uniform, depth uniform in 120-600 pA, i.e. on both sides of delta / 2 = 200 pA, 100 baseline samples either side,
    150 pA raw noise, 100 kHz / 8-pole zero-phase Bessel at 4.17 MHz), timed with CUDA events around each launch after
    a warm-up launch: events/s, sample evaluations/s (window samples x LM trials, an upper bound), LM trials (the
    `iters` column), fraction fitted, median depth error by length and depth class;
  * the TraceAnalyzer step on a 10-minute trace with a share of shallow long events (-180 pA, 9 000-90 000 samples,
    below delta / 2) among two-level events, with stepfit_fallback on and off, alternated.
The card's name and power limit are read in the same run.  Output: one JSON document (stdout and --out).
    python scripts/bench_stepfit_long.py [--events 100000] [--launches 3] [--minutes 10] [--out FILE]"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from cusumtools_b200 import cusum, pipeline, stepfit, synth
from scripts.bench_stepfit import gpu_info


def bench_kernel(n_events: int, launches: int) -> dict:
    dev = torch.device("cuda:0")
    x, off, lens, depth = synth.short_events_device(n_events, dev, seed=2027, min_len=8000, max_len=100_000,
                                                    min_depth=120.0, max_depth=600.0, chunk_events=5000)
    w0, w1 = off[:-1].contiguous(), off[1:].contiguous()
    E = n_events
    tau0 = stepfit.zero_phase_rise_tau(synth.FS, 1e5, 8)
    types0 = torch.full((E,), stepfit.TYPE_STEPFIT_LONG, dtype=torch.int32, device=dev)
    types = types0.clone()
    out = stepfit.StepFitTable(torch.zeros((E, 6), dtype=torch.float64, device=dev),
                               torch.zeros(E, dtype=torch.float64, device=dev), torch.zeros(E, dtype=torch.int32, device=dev),
                               types)
    lv = cusum.LevelTable.empty(E, 3, dev)
    times = []
    for i in range(1 + launches):
        types.copy_(types0)                         # the launch sets every row to 1 / 7: every launch starts alike
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        stepfit.launch_long(x, w0, w1, types, out, lv, padding=synth.SHORT_PAD, tau0=tau0)
        b.record()
        torch.cuda.synchronize()
        if i >= 1:
            times.append(a.elapsed_time(b) * 1e-3)
    t = np.array(times)
    it = out.iters.cpu().numpy()
    st = types.cpu().numpy()
    ln = lens.cpu().numpy()
    win = ln + 2 * synth.SHORT_PAD
    med = float(np.median(t))
    nsamp = int(win.sum())
    # `iters` also counts the few trials that are never evaluated: window samples x iters bounds the passes from above
    sample_trials = float((win.astype(np.float64) * it).sum())
    p = out.params.cpu().numpy()
    dd = np.abs(depth.cpu().numpy())
    by_len = {}
    for lo_, hi_ in ((8000, 16000), (16000, 32000), (32000, 64000), (64000, 100_001)):
        sel = (ln >= lo_) & (ln < hi_)
        res = {}
        for name, dsel in (("below_delta_half", dd < 200.0), ("above_delta_half", dd >= 200.0)):
            m = sel & dsel & (st == 1)
            res[name] = {"events": int((sel & dsel).sum()), "valid_fraction": float(m.sum() / max(1, (sel & dsel).sum())),
                         "median_depth_error": float(np.median(np.abs(np.abs(p[m, 1]) - dd[m]) / dd[m])) if m.any() else None}
        by_len[f"{lo_}-{hi_ - 1}"] = res
    return {"events": E, "window_samples": nsamp, "mean_window": nsamp / E, "launches": launches,
            "kernel_s_median": med, "kernel_s_min": float(t.min()), "kernel_s_max": float(t.max()),
            "events_per_s": E / med, "window_Gsamples_per_s": nsamp / med / 1e9,
            "sample_trials_G_per_s": sample_trials / med / 1e9,
            "lm_trials_mean": float(it.mean()), "lm_trials_max": int(it.max()),
            "fraction_fitted_type1": float(np.mean(st == 1)), "by_length": by_len, "tau0_samples": tau0}


def mixed_trace(n: int, dev):
    """Two-level events and shallow long events (-180 pA) of 9 000 / 20 000 / 45 000 / 90 000 samples, 40 events/s:
    event k takes template k mod 8."""
    tpl = []
    for L in (9000, 20_000, 45_000, 90_000):
        tpl += [synth.EVENT_LEVELS, ((-180.0, L),)]
    return synth.device_trace(n, dev, seed=41, events_per_s=40.0, levels=tpl)


def bench_pipeline(minutes: float, rounds: int) -> dict:
    dev = torch.device("cuda:0")
    n = int(minutes * 60 * synth.FS) // (1 << 16) * (1 << 16)
    codes = mixed_trace(n, dev)
    kw = dict(threshold=5.0, hysteresis=1.0, baseline_block=1 << 16, baseline_min=4900.0, baseline_max=5100.0,
              cusum_delta=400.0, cusum_h=10.0)
    ans = {"off": pipeline.TraceAnalyzer(n, synth.CHIMERA_SETTINGS, 1e5, 8, device=dev, **kw),
           "on": pipeline.TraceAnalyzer(n, synth.CHIMERA_SETTINGS, 1e5, 8, device=dev, stepfit_fallback=True, **kw)}
    for an in ans.values():                         # warm-up (and buffer growth to the event count)
        an.run(codes); torch.cuda.synchronize()
    times = {"off": [], "on": []}
    counts = {}
    for _ in range(rounds):
        for name, an in ans.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = an.run(codes)
            torch.cuda.synchronize()
            times[name].append(time.perf_counter() - t0)
            h = an.tables_to_host(r)
            t = h["types"].astype(np.int64).copy()
            fit = np.isin(t, (0, 1))
            t[fit & (h["overflow"] != 0)] = 6
            t[fit & (h["overflow"] == 0) & (h["n_levels"] < 3)] = 5
            counts[name] = np.bincount(t, minlength=9).tolist()
    return {"samples": n, "minutes": n / synth.FS / 60,
            "template": "cycle of two-level events (-800 / -1600 pA, 1000 + 1000 samples) and one-level -180 pA events "
                        "of 9000 / 20000 / 45000 / 90000 samples, 40 events/s",
            "rounds": rounds, "step_s_off": times["off"], "step_s_on": times["on"],
            "step_s_off_median": float(np.median(times["off"])), "step_s_on_median": float(np.median(times["on"])),
            "final_type_counts_off": counts["off"], "final_type_counts_on": counts["on"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--events", type=int, default=100_000)
    ap.add_argument("--launches", type=int, default=3)
    ap.add_argument("--minutes", type=float, default=10.0)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_stepfit_long.py needs a CUDA device")
    res = {"gpu": gpu_info(), "kernel": bench_kernel(a.events, a.launches)}
    torch.cuda.empty_cache()
    if a.minutes > 0:
        res["pipeline"] = bench_pipeline(a.minutes, a.rounds)
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
