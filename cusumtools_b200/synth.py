"""Synthetic Chimera traces with injected events (SURVEY.md section 8d): the inputs of the
tests and of bench.py.  Not on the hot path; the device generator is torch plumbing so
that multi-gigasample traces never exist on the host."""
from __future__ import annotations

import numpy as np

FS = 4166666.0

#: typical Chimera VC100 settings (the reference only names the keys, plot-trace.py:273-279)
CHIMERA_SETTINGS = {
    "ADCSAMPLERATE": np.array([[4166666.67]]),
    "SETUP_ADCBITS": np.array([[14]]),
    "SETUP_ADCVREF": np.array([[2.5]]),
    "SETUP_TIAgain": np.array([[100e6]]),
    "SETUP_preADCgain": np.array([[1.305]]),
    "SETUP_pAoffset": np.array([[0.0]]),
    "SETUP_mVoffset": np.array([[0.0]]),
}

BASELINE_PA = 5000.0
NOISE_PA = 150.0
EVENT_PERIOD = 4000          # samples between event starts (1 000 events/s at 4.17 MHz -> 4166)
EVENT_LEVELS = ((-800.0, 1000), (-1600.0, 1000))   # (depth pA, samples) two-level template


def _affine(settings):
    vref = float(np.squeeze(settings["SETUP_ADCVREF"]))
    gain = float(np.squeeze(settings["SETUP_TIAgain"])) * float(np.squeeze(settings["SETUP_preADCgain"]))
    off = float(np.squeeze(settings["SETUP_pAoffset"]))
    alpha = 2.0 * vref / 65536.0 / gain * 1e12
    beta = (-vref / gain + off) * 1e12
    return alpha, beta


def quantise(current_pA: np.ndarray, settings=CHIMERA_SETTINGS) -> np.ndarray:
    """Invert scale_raw_data (plot-trace.py:283-287): pA -> uint16 codes with the low
    16-ADCBITS bits zero, clipped to the ADC range."""
    alpha, beta = _affine(settings)
    bits = int(np.squeeze(settings["SETUP_ADCBITS"]))
    step = 1 << (16 - bits)
    c = np.rint((current_pA - beta) / alpha / step) * step
    return np.clip(c, 0, 65536 - step).astype(np.uint16)


def event_starts(n_events: int, period: int = EVENT_PERIOD) -> np.ndarray:
    return 1000 + period * np.arange(n_events, dtype=np.int64) + 500


def c1_trace(n: int = 4166666, n_events: int = 1000, seed: int = 0, settings=CHIMERA_SETTINGS):
    """Config C1: 1 s at 4.17 MHz, baseline +5000 pA, sigma 150 pA white noise, 1000
    two-level events (-800 pA then -1600 pA, 1000 samples each).  Returns (codes uint16,
    true event starts)."""
    rng = np.random.default_rng(seed)
    cur = BASELINE_PA + NOISE_PA * rng.standard_normal(n)
    starts = event_starts(n_events)
    starts = starts[starts + 2000 < n]
    for s in starts:
        o = int(s)
        for depth, length in EVENT_LEVELS:
            cur[o:o + length] += depth
            o += length
    return quantise(cur, settings), starts


def device_trace(n: int, device, seed: int = 1234, events_per_s: float = 1000.0, jitter: int = 500,
                 settings=CHIMERA_SETTINGS, chunk: int = 1 << 26, start_index: int = 0, levels=None):
    """Configs C2/C5: the same signal model generated on the GPU in chunks (Philox),
    events every fs/events_per_s samples with uniform +-jitter on the start.  Returns a
    uint16 CUDA tensor.  `start_index` is the global index of sample 0 (time sharding):
    the event grid is global, the noise stream is per shard (seed).  `levels`: the event
    template as ((depth pA, samples), ...), default EVENT_LEVELS (e.g. ((-1000.0, 100),) for
    short single-level pulses), or a sequence of such templates: event k takes template
    k mod len(levels) (mixed traces: two-level events, short pulses, shallow long events)."""
    if levels is None:
        levels = EVENT_LEVELS
    templates = ([levels] if np.ndim(levels[0]) == 1 else list(levels))
    templates = [tuple((float(d), int(l)) for d, l in tpl) for tpl in templates]
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    alpha, beta = _affine(settings)
    bits = int(np.squeeze(settings["SETUP_ADCBITS"]))
    step = 1 << (16 - bits)
    period = int(round(FS / events_per_s))
    out = torch.empty(n, dtype=torch.uint16, device=device)
    tot = max(sum(l for _, l in tpl) for tpl in templates)
    jg = torch.Generator(device="cpu")
    jg.manual_seed(seed + 7919)
    for c0 in range(0, n, chunk):
        c1 = min(n, c0 + chunk)
        cur = torch.randn(c1 - c0, generator=g, device=device, dtype=torch.float32) * NOISE_PA + BASELINE_PA
        gidx = torch.arange(c0 + start_index, c1 + start_index, device=device, dtype=torch.int64)
        # event k starts at 1500 + k*period + jitter_k (jitter from a hash of k, so it is
        # independent of chunking and sharding)
        k = torch.div(gidx - 1500 + jitter, period, rounding_mode="floor")
        for kk in (k, k - 1):
            h = (kk * 2654435761) % 4294967296
            jit = (h % (2 * jitter + 1)) - jitter if jitter > 0 else torch.zeros_like(h)
            st = 1500 + kk * period + jit
            rel = gidx - st
            for j, tpl in enumerate(templates):
                o = 0
                # (one template: no selection term, so the single-template trace is the one it always was)
                sel = (kk >= 0) if len(templates) == 1 else (kk >= 0) & (kk % len(templates) == j)
                for depth, length in tpl:
                    cur += depth * ((rel >= o) & (rel < o + length) & sel)
                    o += length
        code = torch.round((cur - beta) / alpha / step) * step
        out[c0:c1] = code.clamp_(0, 65536 - step).to(torch.int32).to(torch.uint16)
        del cur, gidx, k, code
    assert tot + jitter < period
    return out


def c3_events(n_events: int, seed: int = 2024, min_len: int = 500, max_len: int = 8000, pad: int = 100,
              noise: float = 24.0):
    """Config C3: pre-extracted events in a flat float32 buffer + int64 offsets.  Lengths
    log-uniform in [min_len, max_len], 1-5 sub-levels with depths from {-600..-2200} pA
    (adjacent steps >= 400 pA), `pad` baseline samples each side."""
    rng = np.random.default_rng(seed)
    lens = np.exp(rng.uniform(np.log(min_len), np.log(max_len), n_events)).astype(np.int64)
    offsets = np.zeros(n_events + 1, dtype=np.int64)
    offsets[1:] = np.cumsum(lens + 2 * pad)
    x = (BASELINE_PA + noise * rng.standard_normal(int(offsets[-1]))).astype(np.float32)
    depths = np.array([-600.0, -1000.0, -1400.0, -1800.0, -2200.0])
    nlev = rng.integers(1, 6, n_events)
    for e in range(n_events):
        L = int(lens[e]); k = int(nlev[e])
        cuts = np.linspace(0, L, k + 1).astype(np.int64)
        prev = None
        for i in range(k):
            choices = depths if prev is None else depths[np.abs(depths - prev) >= 400.0]
            d = float(rng.choice(choices)); prev = d
            a = offsets[e] + pad + cuts[i]; b = offsets[e] + pad + cuts[i + 1]
            x[a:b] += np.float32(d)
    return x, offsets, nlev


def c3_events_device(n_events: int, device, seed: int = 2024, min_len: int = 500, max_len: int = 8000,
                     pad: int = 100, noise: float = 24.0, chunk_events: int = 50000):
    """Config C3 generated on the GPU (1M events = 2.2e9 samples never touch the host):
    same distribution as `c3_events`; adjacent sub-levels differ by >= 400 pA by taking the
    depths cyclically with a random stride.  Returns (samples float32, offsets int64,
    n_sublevels int64) as CUDA tensors."""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    u = torch.rand(n_events, generator=g, device=device, dtype=torch.float64)
    lens = torch.exp(u * (np.log(max_len) - np.log(min_len)) + np.log(min_len)).to(torch.int64)
    nlev = torch.randint(1, 6, (n_events,), generator=g, device=device)
    base = torch.randint(0, 5, (n_events,), generator=g, device=device)
    stride = torch.randint(1, 5, (n_events,), generator=g, device=device)
    tot = lens + 2 * pad
    offsets = torch.zeros(n_events + 1, dtype=torch.int64, device=device)
    offsets[1:] = torch.cumsum(tot, 0)
    total = int(offsets[-1].item())
    x = torch.empty(total, dtype=torch.float32, device=device)
    depths = torch.tensor([-600.0, -1000.0, -1400.0, -1800.0, -2200.0], device=device)
    for e0 in range(0, n_events, chunk_events):
        e1 = min(n_events, e0 + chunk_events)
        a, b = int(offsets[e0].item()), int(offsets[e1].item())
        ev = torch.repeat_interleave(torch.arange(e0, e1, device=device), tot[e0:e1])
        r = torch.arange(a, b, device=device) - offsets[ev] - pad
        L = lens[ev]
        inside = (r >= 0) & (r < L)
        lvl = torch.clamp(r * nlev[ev] // torch.clamp(L, min=1), min=0)
        d = depths[(base[ev] + lvl * stride[ev]) % 5]
        seg = torch.randn(b - a, generator=g, device=device, dtype=torch.float32) * noise + BASELINE_PA
        x[a:b] = seg + d * inside
        del ev, r, L, inside, lvl, d, seg
    return x, offsets, nlev


SHORT_PAD = 100              # baseline samples either side of a short event's window
SHORT_GUARD = 400            # extra baseline between the windows of neighbouring events before filtering


def short_events_device(n_events: int, device, seed: int = 77, min_len: int = 20, max_len: int = 400, pad: int = SHORT_PAD,
                        min_depth: float = 300.0, max_depth: float = 2000.0, noise: float = NOISE_PA,
                        cutoff: float = 1e5, order: int = 8, chunk_events: int = 200_000):
    """Short events for the step-response fit: rectangular pulses of log-uniform length in [min_len, max_len]
    samples and blockage depth uniform in [min_depth, max_depth] pA on a baseline of +-5000 pA (the sign drawn per
    event; the pulse moves the current toward zero), sigma = `noise` pA raw white noise, filtered with the
    project's own zero-phase Bessel (ct_filtfilt_f32) at `cutoff` / `order` and FS.  Every event is filtered
    inside a continuous stretch of baseline (its window plus SHORT_GUARD samples each side), then its window of
    `pad` + length + `pad` samples is cut out.  Returns (samples float32 [sum of windows], offsets int64 [E+1],
    lengths int64 [E], depths float64 [E] signed like the baseline) as CUDA tensors."""
    import torch
    from .filters import bessel_filtfilt
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    u = torch.rand(n_events, generator=g, device=device, dtype=torch.float64)
    lens = torch.exp(u * (np.log(max_len) - np.log(min_len)) + np.log(min_len)).to(torch.int64)
    depth = min_depth + (max_depth - min_depth) * torch.rand(n_events, generator=g, device=device, dtype=torch.float64)
    sgn = torch.where(torch.rand(n_events, generator=g, device=device) < 0.5, -1.0, 1.0).to(torch.float64)
    win = lens + 2 * pad
    offsets = torch.zeros(n_events + 1, dtype=torch.int64, device=device)
    offsets[1:] = torch.cumsum(win, 0)
    out = torch.empty(int(offsets[-1].item()), dtype=torch.float32, device=device)
    for e0 in range(0, n_events, chunk_events):
        e1 = min(n_events, e0 + chunk_events)
        seg = win[e0:e1] + 2 * SHORT_GUARD
        soff = torch.zeros(e1 - e0 + 1, dtype=torch.int64, device=device)
        soff[1:] = torch.cumsum(seg, 0)
        m = int(soff[-1].item())
        ev = torch.repeat_interleave(torch.arange(e1 - e0, device=device), seg)
        r = torch.arange(m, device=device) - soff[ev] - SHORT_GUARD - pad          # index relative to the event start
        inside = (r >= 0) & (r < lens[e0 + ev])
        # the trace of a positive baseline; the event's own sign is applied to its window afterwards (the filter is
        # linear with DC gain 1, and the guards keep the neighbours' pulses out of the window)
        z = torch.randn(m, generator=g, device=device, dtype=torch.float32) * noise - depth[e0 + ev].to(torch.float32) * inside
        y = bessel_filtfilt(z.contiguous(), FS, cutoff, order, pad_value=0.0)
        keep = (r >= -pad) & (r < lens[e0 + ev] + pad)
        w = y[keep].to(torch.float64) + BASELINE_PA
        ek = ev[keep]
        out[int(offsets[e0].item()):int(offsets[e1].item())] = (w * sgn[e0 + ek]).to(torch.float32)
        del ev, r, inside, z, y, keep, w, ek
    return out, offsets, lens, depth * sgn
