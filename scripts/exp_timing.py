"""Per-launch CUDA-event timings of the filter passes in different sequences (is a launch slower when it follows
another launch of the same kind / in a long loop?).  Tuning experiment."""
import ctypes as C, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from cusumtools_b200 import _lib, detect, filters, median, synth
from cusumtools_b200.design import bessel_lowpass
n = int(sys.argv[1]) if len(sys.argv) > 1 else 2_499_999_600
S = synth.CHIMERA_SETTINGS; L = _lib.lib()
raw = synth.device_trace(n, "cuda", seed=1234)
out = torch.empty(n, dtype=torch.float32, device="cuda")
mask = filters.chimera_bitmask(S); alpha, _ = filters.chimera_affine(S)
st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
d = bessel_lowpass(8, 2 * 1e5 / synth.FS); coef = filters.make_coef(d); H = filters.warmup_samples(d)
wsb = int(L.ct_filtfilt_workspace_bytes(n, 1000, H)); ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
mm = torch.empty(2 * int(L.ct_filter_summary_count(n, 1000, H)), dtype=torch.float32, device="cuda")
bl = detect.new_baseline(n, 1 << 20, 4700.0, 5300.0, "cuda"); stats = detect.stats_args(bl, origin=0)
c1, c2 = median.code_median(raw, mask)
def fwd(est):
    rc = L.ct_filter_forward_u16(raw.data_ptr(), n, 1000, est, mask, 0.0, C.byref(coef), H, 0, 0, 0, 1, 0, 0, None, 0, 0, ws.data_ptr(), wsb, st); assert rc == 0
def bwd(est):
    rc = L.ct_filter_backward(n, 1000, est, float(alpha), 5000.0, C.byref(coef), H, 0, out.data_ptr(), ws.data_ptr(), wsb, C.byref(stats), mm.data_ptr(), st); assert rc == 0
def seq(name, fns, est):
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(fns) + 1)]
    torch.cuda.synchronize(); evs[0].record()
    for i, f in enumerate(fns):
        f(est); evs[i + 1].record()
    torch.cuda.synchronize()
    print(f"{name:28s}", " ".join(f"{evs[i].elapsed_time(evs[i + 1]):.3f}" for i in range(len(fns))), flush=True)
for est in (float(c1), 40900.0):
    print("subtracted constant", est, "(median", c1, ")")
    fwd(est); bwd(est); torch.cuda.synchronize()
    seq("fwd x10", [fwd] * 10, est)
    seq("bwd x10", [bwd] * 10, est)
    seq("(fwd bwd) x5", [fwd, bwd] * 5, est)
    time.sleep(0.5)
    seq("after 0.5 s idle: fwd x4", [fwd] * 4, est)
