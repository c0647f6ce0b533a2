"""Step-response fit timings on one GPU, in one run:
  * ct_stepfit_batch alone on 1 M short events (synth.short_events_device: pulses of 20-400 samples, log-uniform,
    100 baseline samples either side, 150 pA raw noise, 100 kHz / 8-pole zero-phase Bessel at 4.17 MHz), timed with
    CUDA events around each launch after warm-up: events/s, window samples/s, LM trials (the `iters` column), fraction fitted;
  * the TraceAnalyzer step on a 10-minute trace of short single-level pulses with stepfit on and off, alternated.
The card's name and power limit are read in the same run.  Output: one JSON document (stdout and --out).
    python scripts/bench_stepfit.py [--events 1000000] [--launches 10] [--minutes 10] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from cusumtools_b200 import cusum, pipeline, stepfit, synth


def gpu_info() -> dict:
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = f"not available ({e})"
    return info


def bench_kernel(n_events: int, launches: int) -> dict:
    dev = torch.device("cuda:0")
    x, off, lens, depth = synth.short_events_device(n_events, dev, seed=2026)
    w0, w1 = off[:-1].contiguous(), off[1:].contiguous()
    E = n_events
    tau0 = stepfit.zero_phase_rise_tau(synth.FS, 1e5, 8)
    types0 = torch.full((E,), stepfit.TYPE_STEPFIT, dtype=torch.int32, device=dev)
    types = types0.clone()
    out = stepfit.StepFitTable(torch.zeros((E, 6), dtype=torch.float64, device=dev),
                               torch.zeros(E, dtype=torch.float64, device=dev), torch.zeros(E, dtype=torch.int32, device=dev),
                               types)
    lv = cusum.LevelTable.empty(E, 3, dev)
    times = []
    for i in range(2 + launches):
        types.copy_(types0)                         # the launch marks failed fits in place: every launch starts alike
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        stepfit.launch(x, w0, w1, types, out, lv, padding=synth.SHORT_PAD, tau0=tau0)
        b.record()
        torch.cuda.synchronize()
        if i >= 2:
            times.append(a.elapsed_time(b) * 1e-3)
    t = np.array(times)
    it = out.iters.cpu().numpy()
    st = types.cpu().numpy()
    nsamp = int(off[-1].item())
    med = float(np.median(t))
    ln = lens.cpu().numpy()
    by_len = {}
    for lo_, hi_ in ((20, 60), (60, 100), (100, 200), (200, 401)):
        m = (ln >= lo_) & (ln < hi_) & (st == 1)
        p = out.params.cpu().numpy()[m]
        dd = np.abs(depth.cpu().numpy()[m])
        by_len[f"{lo_}-{hi_ - 1}"] = {"events": int(((ln >= lo_) & (ln < hi_)).sum()),
                                      "median_depth_error": float(np.median(np.abs(np.abs(p[:, 1]) - dd) / dd)) if m.any() else None}
    return {"events": E, "window_samples": nsamp, "mean_window": nsamp / E, "launches": launches,
            "kernel_s_median": med, "kernel_s_min": float(t.min()), "kernel_s_max": float(t.max()),
            "events_per_s": E / med, "window_Msamples_per_s": nsamp / med / 1e6,
            "lm_evaluations_mean": float(it.mean()), "lm_evaluations_median": float(np.median(it)), "lm_evaluations_max": int(it.max()),
            "fraction_fitted_type1": float(np.mean(st == 1)), "depth_error_by_length": by_len, "tau0_samples": tau0}


def bench_pipeline(minutes: float, rounds: int) -> dict:
    dev = torch.device("cuda:0")
    n = int(minutes * 60 * synth.FS) // (1 << 16) * (1 << 16)
    codes = synth.device_trace(n, dev, seed=31, levels=((-1000.0, 150),))
    kw = dict(threshold=5.0, hysteresis=1.0, baseline_block=1 << 16, baseline_min=4700.0, baseline_max=5300.0,
              cusum_delta=400.0, cusum_h=10.0)
    ans = {"off": pipeline.TraceAnalyzer(n, synth.CHIMERA_SETTINGS, 1e5, 8, device=dev, **kw),
           "on": pipeline.TraceAnalyzer(n, synth.CHIMERA_SETTINGS, 1e5, 8, device=dev, stepfit_samples=500, **kw)}
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
            counts[name] = np.bincount(r.types.cpu().numpy(), minlength=8).tolist()
    return {"samples": n, "minutes": n / synth.FS / 60, "template": "one level, -1000 pA, 150 samples, 1000 events/s",
            "stepfit_samples": 500, "rounds": rounds, "step_s_off": times["off"], "step_s_on": times["on"],
            "step_s_off_median": float(np.median(times["off"])), "step_s_on_median": float(np.median(times["on"])),
            "type_counts_off": counts["off"], "type_counts_on": counts["on"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--events", type=int, default=1_000_000)
    ap.add_argument("--launches", type=int, default=10)
    ap.add_argument("--minutes", type=float, default=10.0)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_stepfit.py needs a CUDA device")
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
