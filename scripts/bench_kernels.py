"""Kernel-by-kernel timing of stage 1-2 on a C2-style device-resident trace (CUDA events on the launching
stream, warm-up first): forward pass, backward pass with / without the fused block sums and chunk extrema,
exact-median count, detection with / without the chunk extrema.  For tuning; bench.py reports the step.

    python scripts/bench_kernels.py [n_samples] [cutoff_hz,...]
"""
import ctypes as C
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from cusumtools_b200 import _lib, detect, filters, median, synth
from cusumtools_b200.design import bessel_lowpass

n = int(sys.argv[1]) if len(sys.argv) > 1 else 2_499_999_600
cutoffs = [float(v) for v in sys.argv[2].split(",")] if len(sys.argv) > 2 else [1e5]
PEAK = 6559.7
S = synth.CHIMERA_SETTINGS
L = _lib.lib()
raw = synth.device_trace(n, "cuda", seed=1234)
out = torch.empty(n, dtype=torch.float32, device="cuda")
mask = filters.chimera_bitmask(S)
alpha, _ = filters.chimera_affine(S)
st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
BLOCK = 1 << 20


def timed(fn, iters=5):
    fn(); fn()
    torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def report(name, ms, bytes_per_sample):
    print(f"  {name:46s} {ms:7.3f} ms  {n / ms / 1e6:7.1f} Gs/s  {bytes_per_sample * n / ms / 1e6:6.0f} GB/s algorithmic "
          f"= {bytes_per_sample * n / ms / 1e6 / PEAK:.3f} of {PEAK:.0f}", flush=True)


c1, c2 = median.code_median(raw, mask)
est = float(c1)
offset = float(filters.scale_codes_host(np.array([c1], dtype=np.uint16), S)[0])
for cutoff in cutoffs:
    d = bessel_lowpass(8, 2 * cutoff / synth.FS)
    coef = filters.make_coef(d)
    H = filters.warmup_samples(d)
    D = filters.scratch_decimation(d, 1000)
    wsb = int(L.ct_filtfilt_workspace_bytes(n, 1000, H))
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    mm = torch.empty(2 * int(L.ct_filter_summary_count(n, 1000, H)), dtype=torch.float32, device="cuda")
    bl = detect.new_baseline(n, BLOCK, 4700.0, 5300.0, "cuda")
    stats = detect.stats_args(bl, origin=0)
    print(f"cutoff {cutoff:.0f} Hz: warm-up {H} samples, scratch keeps every {D}-th forward sample, n = {n}")

    def fwd():
        rc = L.ct_filter_forward_u16(raw.data_ptr(), n, 1000, est, mask, 0.0, C.byref(coef), H, 0, 0, 0, 1, 0, 0, None, 0, 0,
                                     ws.data_ptr(), wsb, st)
        assert rc == 0, L.ct_last_error()

    def bwd(stats_p, mm_p):
        def f():
            rc = L.ct_filter_backward(n, 1000, est, float(alpha), offset, C.byref(coef), H, 0, out.data_ptr(), ws.data_ptr(), wsb,
                                      stats_p, mm_p, st)
            assert rc == 0, L.ct_last_error()
        return f

    if os.environ.get("CT_CLOCKS"):
        # sustained loops with nvidia-smi sampling: do the kernels hold the clock they show in a 5-launch burst?
        import subprocess, time
        for name, fn in (("forward", fwd), ("backward+sums+extrema", bwd(C.byref(stats), mm.data_ptr()))):
            pr = subprocess.Popen(["nvidia-smi", "--query-gpu=clocks.sm,clocks.mem,power.draw,clocks_event_reasons.sw_power_cap,"
                                   "clocks_event_reasons.hw_slowdown,clocks_event_reasons.sw_thermal_slowdown",
                                   "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE, text=True)
            time.sleep(0.2)
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(300):
                fn()
            e1.record(); torch.cuda.synchronize()
            pr.terminate()
            rows = [r.strip() for r in pr.stdout.read().splitlines() if r.strip()]
            print(f"  sustained {name}: {e0.elapsed_time(e1) / 300:.3f} ms per launch over 300 launches; nvidia-smi samples "
                  f"(sm MHz, mem MHz, W, power cap, hw slowdown, thermal): first {rows[:2]} ... mid {rows[len(rows)//2:len(rows)//2+3]} ... last {rows[-2:]}", flush=True)
    t_f = timed(fwd)
    report("forward pass", t_f, 2.0 + 4.0 / D)
    cnt9 = torch.zeros(9, dtype=torch.int64, device="cuda")

    def fwd_count():
        rc = L.ct_filter_forward_u16(raw.data_ptr(), n, 1000, est, mask, 0.0, C.byref(coef), H, 0, 0, max(0, int(c1) - 12), 4, 0, n,
                                     cnt9.data_ptr(), 0, 0, ws.data_ptr(), wsb, st)
        assert rc == 0, L.ct_last_error()

    report("forward pass + fused exact-median window count", timed(fwd_count), 2.0 + 4.0 / D)
    t_b = timed(bwd(None, None))
    report("backward pass", t_b, 4.0 + 4.0 / D)
    t_bs = timed(bwd(C.byref(stats), None))
    report("backward pass + block sums", t_bs, 4.0 + 4.0 / D)
    t_bm = timed(bwd(None, mm.data_ptr()))
    report("backward pass + chunk extrema", t_bm, 4.0 + 4.0 / D)
    t_bsm = timed(bwd(C.byref(stats), mm.data_ptr()))
    report("backward pass + block sums + chunk extrema", t_bsm, 4.0 + 4.0 / D)
    report("PAIR (forward + backward), 6 B/sample", t_f + t_b, 6.0)
    report("PAIR as the step runs it, 6 B/sample", t_f + t_bsm, 6.0)
    if cutoff == cutoffs[0]:
        detect.finish_baseline(bl, 5.0, 1.0)
        cnt = torch.zeros(9, dtype=torch.int64, device="cuda")
        lo = max(0, int(c1) - 4)
        report("exact-median window count (4 codes)", timed(lambda: L.ct_count_window4_u16(raw.data_ptr(), n, mask, lo, 4, cnt.data_ptr(), st)), 2.0)
        report("exact-median window count (8 codes)", timed(lambda: L.ct_count_window_u16(raw.data_ptr(), n, mask, lo, 4, cnt.data_ptr(), st)), 2.0)
        ev0 = detect.detect_events(out, bl)
        ev1 = detect.detect_events(out, bl, chunk_minmax=mm)
        same = torch.equal(ev0.starts, ev1.starts) and torch.equal(ev0.ends, ev1.ends)
        print(f"  detection: {len(ev0)} events; with chunk extrema identical: {same}")
        report("detection (reads the trace)", timed(lambda: detect.detect_events(out, bl)), 4.0)
        report("detection (chunk extrema)", timed(lambda: detect.detect_events(out, bl, chunk_minmax=mm)), 4.0)
    del ws, mm
