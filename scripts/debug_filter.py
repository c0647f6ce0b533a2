import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from cusumtools_b200 import filters, median, synth
from oracle import trace_oracle as to
S = synth.CHIMERA_SETTINGS
for n, ne in ((300000, 70), (24001, 5), (5000, 1)):
    codes, _ = synth.c1_trace(n=n, n_events=ne, seed=0)
    want = to.filter_data(to.scale_raw_data(codes, S), synth.FS, 1e5, 8)
    raw = torch.from_numpy(codes).cuda()
    mask = filters.chimera_bitmask(S)
    c1, c2 = median.code_median(raw, mask)
    srt = np.sort(codes & mask)
    print("n", n, "median codes", c1, c2, "true", srt[(n - 1) // 2], srt[n // 2])
    y = filters.dequant_filtfilt(raw, S, 1e5, 8).cpu().numpy()
    err = np.abs(y - want)
    print("  max err", err.max(), "at", err.argmax(), "mean err", err.mean())
    bad = np.nonzero(err > 0.05)[0]
    print("  bad count", bad.size, "first", bad[:5], "last", bad[-5:])
    for seg in range(0, n, 4096):
        e = err[seg:seg + 4096]
        if e.max() > 0.05:
            print("   seg", seg // 4096, "max", e.max(), "argmax", e.argmax(), "nbad", (e > 0.05).sum())
            break
    print("  y[:4]", y[:4], "want[:4]", want[:4], "y[-4:]", y[-4:], "want[-4:]", want[-4:])
