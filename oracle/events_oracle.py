"""TEST INFRASTRUCTURE — NumPy DEFINITION of stages 2 and 3 (threshold detection, CUSUM+).

The reference repo contains no implementation of these stages: it only consumes their
output (`plot-trace.py:172-203,350-414`, `readevents.py:843-854,1297-1343,1470-1508`) and
converts MOSAIC output into the same table (`mosaicConverter.py:72-194`).  Per
BASELINE.json's north_star this module IS the reference for them: a NumPy implementation
of the published two-sided CUSUM recurrence (Raillon et al., Nanoscale 4 (2012); SURVEY.md
Appendix C) and of the threshold/hysteresis semantics the consumers draw
(`plot-trace.py:379-414`).  Parity status: unpinned by reference tests (there are none).

Design rule that makes "bit-exact indices" meaningful on a GPU: every REDUCTION (block
sums, prefix sums, running minima) is over exactly-defined integers, so its value does not
depend on summation order; every per-sample floating-point step is a fixed sequence of
individually rounded IEEE operations (no fused multiply-add), which numpy, C
(-ffp-contract=off) and CUDA (__fmul_rn/__fsub_rn/__fdiv_rn ...) all evaluate identically.
"""
from __future__ import annotations

import math

import numpy as np

# ------------------------------------------------------------------ stage 2: baseline
STATS_MAX_SHIFT = 8


def stats_shift(half_width: float, block: int) -> int:
    """Fixed-point fraction bits for block statistics: the largest s <= 8 such that
    (half_width * 2^s)^2 * block < 2^62 (int64 sum of squares cannot overflow)."""
    s = STATS_MAX_SHIFT
    while s > -32 and (float(half_width) * 2.0 ** s + 1.0) ** 2 * float(block) >= 2.0 ** 62:
        s -= 1
    return s


STATS_CHUNK = 64


def block_stats(y, block, bmin, bmax, c0, shift):
    """Per-block count / sum / sum of squares of q = rint((y - c0) * 2^shift) over the baseline samples of the
    block.  A sample counts when its whole CHUNK - the aligned group of 64 samples it belongs to, counted from
    sample 0 (the last chunk of the trace may be shorter) - lies inside [bmin, bmax]: a chunk that holds an event
    edge or an excursion is left out as a whole.  `block` is a multiple of 64.  Returns three int64 arrays of
    length ceil(N/block)."""
    y = np.asarray(y, dtype=np.float32)
    n = y.size
    assert block % STATS_CHUNK == 0
    nb = (n + block - 1) // block
    cnt = np.zeros(nb, dtype=np.int64)
    s1 = np.zeros(nb, dtype=np.int64)
    s2 = np.zeros(nb, dtype=np.int64)
    scale = np.float32(2.0 ** shift)
    lo, hi = np.float32(bmin), np.float32(bmax)
    for k in range(nb):
        seg = y[k * block:(k + 1) * block]
        nch = (seg.size + STATS_CHUNK - 1) // STATS_CHUNK
        ok = np.zeros(seg.size, dtype=bool)
        for c in range(nch):
            ch = seg[c * STATS_CHUNK:(c + 1) * STATS_CHUNK]
            if ch.min() >= lo and ch.max() <= hi:
                ok[c * STATS_CHUNK:(c + 1) * STATS_CHUNK] = True
        d = (seg[ok] - np.float32(c0)).astype(np.float32) * scale
        q = np.rint(d).astype(np.int64)
        cnt[k] = q.size
        s1[k] = q.sum()
        s2[k] = (q * q).sum()
    return cnt, s1, s2


def block_stats_fast(y, block, bmin, bmax, c0, shift):
    """`block_stats`, vectorised over chunks (same definition; tests assert the identity)."""
    y = np.asarray(y, dtype=np.float32)
    n = y.size
    assert block % STATS_CHUNK == 0
    nb = (n + block - 1) // block
    nfull = n // STATS_CHUNK
    lo, hi = np.float32(bmin), np.float32(bmax)
    ch = y[:nfull * STATS_CHUNK].reshape(nfull, STATS_CHUNK)
    ok = (ch.min(axis=1) >= lo) & (ch.max(axis=1) <= hi)
    q = np.rint((ch - np.float32(c0)).astype(np.float32) * np.float32(2.0 ** shift)).astype(np.int64)
    q[~ok] = 0
    c_cnt = np.where(ok, STATS_CHUNK, 0).astype(np.int64)
    c_s1, c_s2 = q.sum(axis=1), (q * q).sum(axis=1)
    tail = y[nfull * STATS_CHUNK:]
    if tail.size:
        t_ok = tail.min() >= lo and tail.max() <= hi
        tq = np.rint((tail - np.float32(c0)).astype(np.float32) * np.float32(2.0 ** shift)).astype(np.int64) if t_ok else np.zeros(0, np.int64)
        c_cnt = np.append(c_cnt, tq.size); c_s1 = np.append(c_s1, tq.sum()); c_s2 = np.append(c_s2, (tq * tq).sum())
    cpb = block // STATS_CHUNK
    pad = nb * cpb - c_cnt.size
    if pad:
        z = np.zeros(pad, np.int64)
        c_cnt, c_s1, c_s2 = np.append(c_cnt, z), np.append(c_s1, z), np.append(c_s2, z)
    return (c_cnt.reshape(nb, cpb).sum(axis=1), c_s1.reshape(nb, cpb).sum(axis=1), c_s2.reshape(nb, cpb).sum(axis=1))


def baseline_from_stats(cnt, s1, s2, c0, shift, min_count=16):
    """Block mean / population std from the exact integer sums, as a fixed sequence of
    individually rounded float64 operations (so numpy, C and CUDA agree bit for bit):
      ma = s1/cnt ; mean = c0 + ma*2^-shift ; var = s2/cnt - ma*ma ;
      std = sqrt(max(var, 0))*2^-shift.
    Blocks with fewer than `min_count` in-window samples inherit the nearest earlier valid
    block (or the first valid one)."""
    cnt = np.asarray(cnt, np.int64)
    nb = len(cnt)
    c = cnt.astype(np.float64)
    ok = cnt >= min_count
    cs = np.where(ok, c, 1.0)
    inv = 2.0 ** (-shift)
    ma = np.asarray(s1, np.int64).astype(np.float64) / cs
    mean = float(np.float32(c0)) + ma * inv
    var = np.asarray(s2, np.int64).astype(np.float64) / cs - ma * ma
    std = np.sqrt(np.where(var > 0, var, 0.0)) * inv
    mean = np.where(ok, mean, np.nan)
    std = np.where(ok, std, np.nan)
    valid = np.nonzero(ok)[0]
    if valid.size == 0:
        raise ValueError("no baseline block has enough samples inside [baseline_min, baseline_max]")
    last = valid[0]
    for k in range(nb):
        if not ok[k]:
            mean[k], std[k] = mean[last], std[last]
        else:
            last = k
    return mean, std


def thresholds(mean, std, threshold, hysteresis):
    """plot-trace.py:408-411: sign = sign(baseline); start line = baseline - sign*threshold*
    stdev, end line = baseline - sign*(threshold - hysteresis)*stdev.  Rounded to float32,
    the type they are compared in."""
    sign = np.where(np.asarray(mean) >= 0, 1, -1).astype(np.int32)
    t_start = (mean - sign * threshold * std).astype(np.float32)
    t_end = (mean - sign * (threshold - hysteresis) * std).astype(np.float32)
    return sign, t_start, t_end


# ----------------------------------------------------------------- stage 2: detection
def detect_events(y, block, sign, t_start, t_end, state_in=False):
    """Threshold/hysteresis event detection.

    Sequential definition: walking the samples in order, an event STARTS at the first
    sample beyond the start line while outside an event and ENDS at the first sample back
    beyond the end line while inside one; the event occupies [start, end).  Returns
    (starts int64[E], ends int64[E], open_start) where open_start is the start index of an
    event still open at the end of the data (or -1).

    Precondition: sign*t_start <= sign*t_end in every block (hysteresis >= 0).  With crossed
    lines a sample between them is both beyond the start line and back beyond the end line,
    and this vectorised form no longer agrees with `detect_events_sequential`."""
    y = np.asarray(y, dtype=np.float32)
    n = y.size
    if n == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64), -1
    blk = np.arange(n, dtype=np.int64) // block
    pos = np.asarray(sign)[blk] > 0
    ts = np.asarray(t_start, dtype=np.float32)[blk]
    te = np.asarray(t_end, dtype=np.float32)[blk]
    a = np.where(pos, y < ts, y > ts)
    b = np.where(pos, y > te, y < te)
    sym = np.where(a, 1, np.where(b, 2, 0)).astype(np.int8)
    idx = np.where(sym != 0, np.arange(n, dtype=np.int64), -1)
    last = np.maximum.accumulate(idx)
    filled = np.where(last >= 0, sym[np.maximum(last, 0)], 1 if state_in else 2)
    inside = filled == 1
    prev = np.concatenate(([bool(state_in)], inside[:-1]))
    starts = np.nonzero(inside & ~prev)[0].astype(np.int64)
    ends = np.nonzero(~inside & prev)[0].astype(np.int64)
    open_start = -1
    if state_in:
        # the first end closes an event opened before this data
        ends = ends[1:] if ends.size and (starts.size == 0 or ends[0] < starts[0]) else ends
    if starts.size > ends.size:
        open_start = int(starts[-1])
        starts = starts[:-1]
    return starts, ends, open_start


def detect_events_sequential(y, block, sign, t_start, t_end, state_in=False):
    """The literal state machine (pure Python, small inputs): the definition
    `detect_events` vectorises."""
    starts, ends = [], []
    inside = bool(state_in)
    start = -1
    for n in range(len(y)):
        k = n // block
        v = np.float32(y[n])
        if sign[k] > 0:
            a, b = v < np.float32(t_start[k]), v > np.float32(t_end[k])
        else:
            a, b = v > np.float32(t_start[k]), v < np.float32(t_end[k])
        if not inside and a:
            inside, start = True, n
        elif inside and b:
            inside = False
            if start >= 0:
                starts.append(start); ends.append(n)
    return (np.array(starts, np.int64), np.array(ends, np.int64), start if inside else -1)


def intra_crossings(x, local_baseline, local_stdev, intra_threshold, intra_hysteresis):
    """Intra-event threshold crossings of one event window (consumer side: readevents.py:1340-1343 reads
    rate.csv's `intra_crossing_times_us` as start/end pairs and shades them, :1363-1366 draws the lines
    local_baseline - intra_threshold*local_stdev and local_baseline - (intra_threshold -
    intra_hysteresis)*local_stdev, sign-mirrored; the thresholds come from summary.txt, :73-79).

    Definition: the detector's own automaton (`detect_events`) over the window samples with those two
    lines (float32, `thresholds`), starting outside; a crossing still open at the end of the window ends
    there.  Returns int64 [C, 2] (start, end) sample indices relative to the window start."""
    x = np.asarray(x, dtype=np.float32)
    sign, ts, te = thresholds(np.array([float(local_baseline)]), np.array([float(local_stdev)]), intra_threshold, intra_hysteresis)
    s, e, open_start = detect_events(x, max(1, x.size), sign, ts, te)
    if open_start >= 0:
        s, e = np.append(s, open_start), np.append(e, x.size)
    return np.stack((s, e), axis=1).astype(np.int64) if s.size else np.zeros((0, 2), np.int64)


def event_windows(starts, ends, n, padding, minpoints, maxpoints):
    """Event sample windows handed to CUSUM+: [start - padding, end + padding), and the
    `type` column of rate.csv (plot-trace.py:354-357: 0/1 accepted, >1 rejected):
      0 accepted; 2 shorter than minpoints; 3 longer than maxpoints;
      4 padding window leaves the trace or overlaps a neighbouring event."""
    starts = np.asarray(starts, np.int64)
    ends = np.asarray(ends, np.int64)
    w0 = starts - padding
    w1 = ends + padding
    typ = np.zeros(starts.size, dtype=np.int32)
    length = ends - starts
    prev_end = np.concatenate(([0], ends[:-1]))
    next_start = np.concatenate((starts[1:], [n]))
    bad_pad = (w0 < prev_end) | (w1 > next_start) | (w0 < 0) | (w1 > n)
    typ[bad_pad] = 4
    typ[length > maxpoints] = 3
    typ[length < minpoints] = 2
    return w0, w1, typ


# ------------------------------------------------------------------- stage 3: CUSUM+
CUSUM_Q = np.float32(64.0)          # samples are quantised to 1/64 pA
CUSUM_SSCALE = np.float32(1024.0)   # log-likelihood increments quantised to 2^-10
CUSUM_SMAX = np.float32(2097152.0)   # |s| <= 2^21 fixed-point units (2048 nats per sample)


def cusum_quantise(x):
    """q_k = rint((x_k - x_0) * 64) as int32 (the conversion saturates at the int32 range); int64 array."""
    x = np.asarray(x, dtype=np.float32)
    d = (x - x[0]).astype(np.float32) * CUSUM_Q
    return np.clip(np.rint(d), -2147483648.0, 2147483647.0).astype(np.int64)


def cusum_increments(q, k0, delta):
    """Fixed-point log-likelihood-ratio increments s+_k, s-_k for k in (k0, n) with the running mean / population
    variance of the current level taken over q[k0..k] (SURVEY.md Appendix C).  The sums are exact integers of the
    deviations from the anchor sample, d_j = q_j - q_k0 (small numbers, so that float32 carries everything that
    follows; order independent, so a parallel scan gives the same values); per sample, in this exact order of
    individually rounded float32 operations:
      cnt  = k - k0 + 1 ;  rc = 1.0f / (float)cnt
      m    = (float)Sd * rc                                (Sd = sum of d over [k0, k], int64 -> float32, RN)
      v    = (float)Sdd * rc - m * m                       (three operations; Sdd = sum of d^2)
      if !(v > 0): s+ = s- = 0
      r    = dq * (1.0f / v)                               (dq = delta*64; correctly rounded reciprocal)
      t    = (float)d_k - m
      s+   = rint(clamp(( r) * (t - dq/2) * 1024))
      s-   = rint(clamp((-r) * (t + dq/2) * 1024))
    """
    q = np.asarray(q, dtype=np.int64)
    seg = q[k0:] - q[k0]
    Sd = np.cumsum(seg)[1:]
    Sdd = np.cumsum(seg * seg)[1:]
    cnt = np.arange(2, seg.size + 1, dtype=np.int64)
    dq = np.float32(np.float32(delta) * CUSUM_Q)
    hq = np.float32(dq * np.float32(0.5))
    one = np.float32(1.0)
    rc = (one / cnt.astype(np.float32)).astype(np.float32)
    m = (Sd.astype(np.float32) * rc).astype(np.float32)
    v = ((Sdd.astype(np.float32) * rc).astype(np.float32) - (m * m).astype(np.float32)).astype(np.float32)
    ok = v > 0
    vs = np.where(ok, v, one).astype(np.float32)
    r = (dq * (one / vs).astype(np.float32)).astype(np.float32)
    t = (seg[1:].astype(np.float32) - m).astype(np.float32)
    sp = (r * (t - hq).astype(np.float32)).astype(np.float32) * CUSUM_SSCALE
    sn = ((-r) * (t + hq).astype(np.float32)).astype(np.float32) * CUSUM_SSCALE
    sp = np.minimum(np.maximum(sp, -CUSUM_SMAX), CUSUM_SMAX)
    sn = np.minimum(np.maximum(sn, -CUSUM_SMAX), CUSUM_SMAX)
    spi = np.where(ok, np.rint(sp), 0).astype(np.int64)
    sni = np.where(ok, np.rint(sn), 0).astype(np.int64)
    return spi, sni


def cusum_event(x, delta, h, max_levels=32):
    """Two-sided CUSUM+ segmentation of one event window x[0..n).

    Returns (edges int64[L+1], overflow) with edges[0] = 0, edges[L] = n: level i is
    x[edges[i] : edges[i+1]].  With S± the exact integer cumulative sums of s± from the
    anchor (S = 0 at the anchor) and g± = S± - running min of S±, a jump is detected at the
    first k with g+ > H or g- > H (H = rint(h*1024)); the test with the larger g wins (ties:
    +); the new level starts one sample after the LAST index at which the winning S attained
    its running minimum; the anchor moves to k (Appendix C) and all sums restart.  At most
    `max_levels` levels are produced; `overflow` says more jumps were pending."""
    q = cusum_quantise(x)
    n = q.size
    H = int(np.rint(np.float32(h) * CUSUM_SSCALE))
    edges = [0]
    k0 = 0
    overflow = False
    while k0 + 1 < n:
        spi, sni = cusum_increments(q, k0, delta)
        Sp = np.concatenate(([0], np.cumsum(spi)))
        Sn = np.concatenate(([0], np.cumsum(sni)))
        gp = Sp - np.minimum.accumulate(Sp)
        gn = Sn - np.minimum.accumulate(Sn)
        hit = np.nonzero((gp > H) | (gn > H))[0]
        if hit.size == 0:
            break
        j = int(hit[0])              # offset from k0 (>= 1)
        S = Sp if gp[j] >= gn[j] else Sn
        mn = S[:j + 1].min()
        jmin = int(np.nonzero(S[:j + 1] == mn)[0][-1])
        if len(edges) >= max_levels:
            overflow = True
            break
        edges.append(k0 + jmin + 1)
        k0 = k0 + j
    edges.append(n)
    return np.array(edges, dtype=np.int64), overflow


def level_stats(x, edges):
    """Per-level length, mean and population standard deviation (pA) from the exact
    integer sums of the quantised samples: mean = x0 + (Sq/len)/64,
    std = sqrt(max(Sqq - Sq*Sq/len, 0)/len)/64 evaluated in float64."""
    x = np.asarray(x, dtype=np.float32)
    q = cusum_quantise(x)
    L = len(edges) - 1
    length = np.diff(edges).astype(np.int64)
    mean = np.empty(L)
    std = np.empty(L)
    x0 = float(x[0])
    for i in range(L):
        seg = q[edges[i]:edges[i + 1]]
        n = float(seg.size)
        a = float(np.float64(int(seg.sum())))
        b = float(np.float64(int((seg * seg).sum())))
        mean[i] = x0 + (a / n) / 64.0
        std[i] = math.sqrt(max(b - a * a / n, 0.0) / n) / 64.0
    return length, mean, std


def cusum_batch(samples, offsets, delta, h, max_levels=32):
    """Batched form over a flat event buffer: event e is samples[offsets[e]:offsets[e+1]].
    Returns n_levels int32[E], edges int32[E, max_levels+1] (unused = -1), mean/std
    float64[E, max_levels], overflow uint8[E]."""
    E = len(offsets) - 1
    nlev = np.zeros(E, dtype=np.int32)
    edges = np.full((E, max_levels + 1), -1, dtype=np.int32)
    mean = np.zeros((E, max_levels))
    std = np.zeros((E, max_levels))
    ovf = np.zeros(E, dtype=np.uint8)
    for e in range(E):
        x = samples[offsets[e]:offsets[e + 1]]
        if len(x) == 0:
            continue
        ed, o = cusum_event(x, delta, h, max_levels)
        _, mu, sd = level_stats(x, ed)
        L = len(ed) - 1
        nlev[e] = L
        edges[e, :L + 1] = ed
        mean[e, :L] = mu
        std[e, :L] = sd
        ovf[e] = o
    return nlev, edges, mean, std, ovf


def cusum_event_sequential(x, delta, h, max_levels=32):
    """The literal sample-by-sample recurrence (pure Python; small inputs).  Uses the
    max-plus form g = max(g + s, 0) and tracks the last reset index, which in exact integer
    arithmetic equals the S - min S form of `cusum_event`."""
    q = cusum_quantise(x)
    n = q.size
    H = int(np.rint(np.float32(h) * CUSUM_SSCALE))
    dq = np.float32(np.float32(delta) * CUSUM_Q)
    hq = np.float32(dq * np.float32(0.5))
    one = np.float32(1.0)
    edges = [0]
    overflow = False
    k0 = 0
    qa = int(q[0])
    Sd = Sdd = 0
    gp = gn = 0
    rp = rn = 0   # last index at which g was (re)set to zero
    k = 1
    while k < n:
        d = int(q[k]) - qa
        Sd += d; Sdd += d * d
        cnt = k - k0 + 1
        rc = np.float32(one / np.float32(cnt))
        m = np.float32(np.float32(Sd) * rc)
        v = np.float32(np.float32(np.float32(Sdd) * rc) - np.float32(m * m))
        sp = sn = 0
        if v > 0:
            r = np.float32(dq * np.float32(one / v))
            t = np.float32(np.float32(d) - m)
            a = np.float32(np.float32(r * np.float32(t - hq)) * CUSUM_SSCALE)
            b = np.float32(np.float32((-r) * np.float32(t + hq)) * CUSUM_SSCALE)
            a = min(max(a, -CUSUM_SMAX), CUSUM_SMAX)
            b = min(max(b, -CUSUM_SMAX), CUSUM_SMAX)
            sp, sn = int(np.rint(a)), int(np.rint(b))
        gp += sp
        if gp <= 0:
            gp, rp = 0, k
        gn += sn
        if gn <= 0:
            gn, rn = 0, k
        if gp > H or gn > H:
            jmin = rp if gp >= gn else rn
            if len(edges) >= max_levels:
                overflow = True
                break
            edges.append(jmin + 1)
            k0 = k
            qa = int(q[k]); Sd = Sdd = 0
            gp = gn = 0
            rp = rn = k
        k += 1
    edges.append(n)
    return np.array(edges, dtype=np.int64), overflow
