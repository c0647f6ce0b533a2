"""Inputs that drive the CUSUM+ kernels (csrc/ct_cusum.cu) down each of their paths, with a host-side witness per case.

Every builder returns a Case: one float32 trace, the event windows into it, the parameters of the batch and a
`witness`, a dict of named facts computed on the host that show the case reaches the path it is named for.  A window
that the kernels reject (empty, reversed, outside the trace, longer than 2^30, type != 0) stands for an empty event,
so `twin(case)` is the C twin of the whole batch row for row.  tests/test_cusum_cases_host.py checks the twin against
the NumPy definition and every witness; tests/test_gpu_cusum_paths.py runs the kernels on the same cases.

The dispatch rule of the kernels, restated (ct_cusum_seq_kernel / cusum_launch):
  * a batch of fewer than SEQ_MIN_EVENTS events, or a trace whose pointer is not 16-byte aligned, goes to the
    warp-per-event kernel whole;
  * otherwise one lane per event takes every accepted window of at most SEQ_MAX samples, and the warps take the longer
    ones (the "pending" list of the workspace).
"""
from __future__ import annotations

import functools
from dataclasses import dataclass, field

import numpy as np

from oracle import c_twin, events_oracle as eo

SEQ_MIN_EVENTS = 16384          # kSeqMinEvents
SEQ_MAX = 16384                 # kSeqMax: longest window one lane takes
SEQ_TAB = 8192 + 16             # kSeqTab: entries of the shared-memory reciprocal table 1.0f / cnt
SMAX = 2 ** 21                  # kSMax: clamp of one fixed-point increment
MAX_WINDOW = 0x3FFFFFFF         # longest window the kernels accept
H_MAX = 2.0 ** 18               # largest accepted h
F32 = np.float32


@dataclass(eq=False)
class Case:
    name: str
    y: np.ndarray               # float32 trace
    w0: np.ndarray              # int64 window starts
    w1: np.ndarray              # int64 window ends
    types: np.ndarray           # int32 rate.csv types (0: CUSUM+ runs)
    delta: float
    h: float
    max_levels: int
    witness: dict = field(default_factory=dict)     # named facts that must all be true
    groups: dict = field(default_factory=dict)      # named row lists the GPU tests look at

    @property
    def n(self) -> int:
        return self.w0.size

    def window(self, i: int) -> np.ndarray:
        return self.y[self.w0[i]:self.w1[i]]


def accepted(y, w0, w1, types) -> np.ndarray:
    """Windows the kernels segment; every other row is left with n_levels 0, overflow 0 and edges -1."""
    ln = w1 - w0
    return (ln > 0) & (w0 >= 0) & (w1 <= y.size) & (ln <= MAX_WINDOW) & (types == 0)


def pending(y, w0, w1, types, n_events: int, aligned16: bool) -> np.ndarray:
    """Rows among the first `n_events` that the lanes leave to the warp kernel, sorted."""
    w0, w1, types = w0[:n_events], w1[:n_events], types[:n_events]
    ok = accepted(y, w0, w1, types)
    if n_events >= SEQ_MIN_EVENTS and aligned16:
        ok &= (w1 - w0) > SEQ_MAX
    return np.nonzero(ok)[0]


def flat(case: Case):
    """The accepted windows back to back (rejected ones empty): the input of the C twin and of the NumPy definition."""
    ok = accepted(case.y, case.w0, case.w1, case.types)
    lens = np.where(ok, case.w1 - case.w0, 0)
    offs = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    parts = [case.y[a:b] for a, b, k in zip(case.w0, case.w1, ok) if k]
    return (np.concatenate(parts) if parts else np.zeros(0, F32)), offs


@functools.lru_cache(maxsize=None)
def _twin(case: Case):
    x, offs = flat(case)
    return c_twin.cusum_batch(x, offs, case.delta, case.h, case.max_levels)


def twin(case: Case):
    """(n_levels, edges, mean, std, overflow) of the C twin for every row of the case."""
    return _twin(case)


def distinct_rows(case: Case):
    """(first, rep): the first row of every distinct accepted window (or of the rejected rows), and for every row the
    first row with the same window.  Identical windows have identical results by definition."""
    ok = accepted(case.y, case.w0, case.w1, case.types)
    key = np.stack((np.where(ok, case.w0, -1), np.where(ok, case.w1, -1)), axis=1)
    _, first, inv = np.unique(key, axis=0, return_index=True, return_inverse=True)
    return np.sort(first), first[inv.ravel()]


def subset(case: Case, rows) -> Case:
    """The case restricted to `rows` (same trace and parameters)."""
    rows = np.asarray(rows)
    return Case(case.name, case.y, case.w0[rows], case.w1[rows], case.types[rows], case.delta, case.h, case.max_levels)


# ---------------------------------------------------------------------------------------------- host arithmetic
def quiet_sums(x) -> np.ndarray:
    """Sd_k = sum of q_j - q_0 over j <= k for one window (the first level, anchor at sample 0)."""
    q = eo.cusum_quantise(x)
    return np.cumsum(q - q[0])


def increment_at(x, k: int, delta: float, rc, clamp: bool = True):
    """(s+, s-) of sample k of a window whose anchor is sample 0, with `rc` in place of 1.0f / (k + 1): the arithmetic of
    events_oracle.cusum_increments for one sample.  Unclamped values are returned as float32."""
    q = eo.cusum_quantise(x[:k + 1])
    d = q - q[0]
    Sd, Sdd = int(d.sum()), int((d * d).sum())
    rc = F32(rc)
    dq = F32(F32(delta) * F32(64.0)); hq = F32(dq * F32(0.5))
    m = F32(F32(Sd) * rc)
    v = F32(F32(F32(Sdd) * rc) - F32(m * m))
    if not v > 0:
        return 0, 0
    r = F32(dq * F32(F32(1.0) / v))
    t = F32(F32(d[-1]) - m)
    a = F32(F32(r * F32(t - hq)) * F32(1024.0))
    b = F32(F32(F32(-r) * F32(t + hq)) * F32(1024.0))
    if not clamp:
        return a, b
    a = min(max(a, -F32(SMAX)), F32(SMAX)); b = min(max(b, -F32(SMAX)), F32(SMAX))
    return int(np.rint(a)), int(np.rint(b))


def first_level_g(x, delta: float):
    """g+_k, g-_k of the first level of a window (anchor at sample 0, no detection assumed), k = 0 .. n-1."""
    sp, sn = eo.cusum_increments(eo.cusum_quantise(x), 0, delta)
    Sp, Sn = np.concatenate(([0], np.cumsum(sp))), np.concatenate(([0], np.cumsum(sn)))
    return Sp - np.minimum.accumulate(Sp), Sn - np.minimum.accumulate(Sn)


def quiet_fraction(x, delta: float) -> float:
    """Share of the samples k >= 1 of a one-level window whose deviation from the running mean lies within +-delta/2
    (t of events_oracle.cusum_increments): the samples the lanes may pass over without evaluating the increments."""
    q = eo.cusum_quantise(x)
    d = q - q[0]
    k = np.arange(1, q.size)
    m = (np.cumsum(d)[1:].astype(F32) * (F32(1.0) / (k + 1).astype(F32))).astype(F32)
    t = (d[1:].astype(F32) - m).astype(F32)
    hq = F32(F32(F32(delta) * F32(64.0)) * F32(0.5))
    return float(np.mean(np.abs(t) <= hq))


def wrap32(v):
    return (np.asarray(v, np.int64) + 2 ** 31) % 2 ** 32 - 2 ** 31


# ------------------------------------------------------------------------------------------------ trace builder
class _Trace:
    """A trace grown segment by segment, and the windows into it."""

    def __init__(self, seed: int):
        self.rng = np.random.default_rng(seed)
        self.parts: list[np.ndarray] = []
        self.size = 0
        self.rows: list[tuple[int, int, int]] = []

    def add(self, x) -> int:
        a = self.size
        self.parts.append(np.asarray(x, np.float64))
        self.size += len(x)
        return a

    def noise(self, n: int, base: float = 5000.0, sigma: float = 24.0) -> np.ndarray:
        return base + sigma * self.rng.standard_normal(n)

    def window(self, a: int, b: int, typ: int = 0) -> int:
        self.rows.append((int(a), int(b), int(typ)))
        return len(self.rows) - 1

    def segment(self, x, typ: int = 0) -> int:
        """x as a window of its own (after a gap of 7 samples, so that window starts fall on every residue)."""
        self.add(self.noise(7))
        a = self.add(x)
        return self.window(a, a + len(x), typ)

    def steps(self, n: int, n_steps: int, depth: float = 900.0, base: float = 5000.0) -> np.ndarray:
        """A window of n samples with n_steps alternating jumps of +-depth at random places."""
        x = self.noise(n, base)
        for j, c in enumerate(np.sort(self.rng.choice(np.arange(10, n - 10), n_steps, replace=False))):
            x[c:] += depth * (-1) ** j
        return x

    def filler(self, rows: int) -> None:
        """`rows` short windows (1-64 samples, drawn from 256 distinct ones in a 4096-sample segment with steps): they
        fill a batch up to the size at which the lanes take it."""
        x = self.noise(4096)
        for c in range(40, 4096, 57):
            x[c:c + 25] -= 800
        a = self.add(x)
        pool = [(a + int(s), a + int(s) + int(L)) for s, L in zip(self.rng.integers(0, 4096 - 64, 256), self.rng.integers(1, 65, 256))]
        for i in range(rows):
            self.window(*pool[i % len(pool)])

    def case(self, name: str, delta: float = 400.0, h: float = 10.0, max_levels: int = 16, min_rows: int = 0) -> Case:
        if min_rows > len(self.rows):
            self.filler(min_rows - len(self.rows))
        w = np.array(self.rows, np.int64).reshape(-1, 3)
        return Case(name, np.concatenate(self.parts).astype(F32), w[:, 0].copy(), w[:, 1].copy(),
                    w[:, 2].astype(np.int32), float(delta), float(h), int(max_levels))


LANES = SEQ_MIN_EVENTS + 37       # rows of a batch the lanes take


# ---------------------------------------------------------------------------------------------------- builders
@functools.lru_cache(maxsize=None)
def dispatch(n_events: int) -> Case:
    """n_events rows (one side or the other of SEQ_MIN_EVENTS) with windows of SEQ_MAX - 1, SEQ_MAX and SEQ_MAX + 1
    samples, longer ones, rejected ones and short filler."""
    T = _Trace(n_events)
    for L in (SEQ_MAX - 1, SEQ_MAX, SEQ_MAX + 1, 20000):
        T.segment(T.steps(L, 3))
    T.segment(T.steps(SEQ_MAX + 1, 2), typ=2)
    T.segment(T.steps(300, 2))
    T.window(100, 100); T.window(200, 150)
    T.filler(n_events - len(T.rows))
    c = T.case(f"dispatch_E{n_events}")
    lens = c.w1 - c.w0
    ok = accepted(c.y, c.w0, c.w1, c.types)
    c.witness = {
        "batch size as named": c.n == n_events,
        "lanes take windows of SEQ_MAX - 1 and SEQ_MAX": bool(np.any(ok & (lens == SEQ_MAX - 1)) and np.any(ok & (lens == SEQ_MAX))),
        "warps take a window of SEQ_MAX + 1": bool(np.any(ok & (lens == SEQ_MAX + 1))),
        "a rejected window of SEQ_MAX + 1": bool(np.any(~ok & (lens == SEQ_MAX + 1))),
        "the three lengths have levels": bool(np.all(twin(c)[0][ok & (abs(lens - SEQ_MAX) <= 1)] >= 3)),
    }
    return c


@functools.lru_cache(maxsize=None)
def line_grid(tail: int) -> Case:
    """Windows starting at every residue mod 32 (the 128-byte line grid the lanes copy), duplicated and overlapping
    windows, and 40 windows of 1-40 samples that end on the last sample of a trace of length = tail (mod 32)."""
    T = _Trace(100 + tail)
    x = T.noise(32 * 400)
    for c in range(0, x.size, 150):
        x[c:c + 70] -= 600 + 5 * (c % 7)
    a = T.add(x)
    dup = []
    for r in range(32):
        for k, L in enumerate((1, 7, 31, 32, 33, 95, 257, 700)):
            s = a + 32 * (r + 40 * k) + r
            T.window(s, s + L)
            if L == 257:
                dup.append(T.window(s, s + L))               # the same window twice
                T.window(s + 100, s + L + 100)               # and one overlapping it
    T.window(a, a + x.size)                                  # overlaps all of them
    T.filler(LANES - len(T.rows) - 40)
    x = T.noise((tail - T.size) % 32 + 64)
    x[-20:] -= 700
    n = T.add(x) + x.size                                    # length of the finished trace
    for L in range(1, 41):
        T.window(n - L, n)
    c = T.case(f"line_grid_tail{tail}")
    c.groups["dup"] = dup
    c.witness = {
        "trace length = tail (mod 32)": c.y.size % 32 == tail,
        "windows start at all 32 residues": set((c.w0 % 32).tolist()) == set(range(32)),
        "windows of 1..40 samples end on the last sample": set((c.w1 - c.w0)[c.w1 == c.y.size].tolist()) >= set(range(1, 41)),
        # whole and partial lines in one round: a window ending on a partial last line also reads whole lines
        "last line partial, read together with whole ones": tail == 0 or bool(np.any((c.w1 == c.y.size) & (c.w1 - c.w0 > tail))),
        "duplicated windows": len(dup) == 32 and all(c.w0[i] == c.w0[i - 1] and c.w1[i] == c.w1[i - 1] for i in dup),
        "windows with levels": int((twin(c)[0] >= 3).sum()) > 200,
    }
    return c


@functools.lru_cache(maxsize=None)
def recip_table() -> Case:
    """Plateaus across the end of the shared reciprocal table (counts up to SEQ_TAB - 1 come from the table, larger
    ones from a division), a plateau longer than the table that ends in a step, and a one-sample spike at count
    SEQ_TAB itself, with h chosen so that the increments computed with 1.0f / SEQ_TAB and with 1.0f / (SEQ_TAB - 1)
    fall on either side of H: whether the spike is detected depends on which reciprocal the kernel uses there."""
    T = _Trace(7)
    plateaus = [T.segment(T.noise(L)) for L in (8207, 8208, 8209, 8217, 9000, 16384)]
    x = T.noise(SEQ_TAB + 300)
    x[SEQ_TAB + 100:] -= 1000
    stepped = T.segment(x)
    for amp in np.arange(300.0, 400.0, 3.0):
        x = T.noise(9000)
        x[SEQ_TAB - 1] += amp
        xs = x.astype(F32)
        s_tab, s_div = increment_at(xs, SEQ_TAB - 1, 400.0, F32(1.0) / F32(SEQ_TAB)), increment_at(xs, SEQ_TAB - 1, 400.0, F32(1.0) / F32(SEQ_TAB - 1))
        if s_tab[0] != s_div[0]:
            break
    H = min(s_tab[0], s_div[0])
    spike = T.segment(x)
    c = T.case("recip_table", h=H / 1024.0, min_rows=LANES)
    nl, ed = twin(c)[0], twin(c)[1]
    sp, _ = eo.cusum_increments(eo.cusum_quantise(c.window(spike)), 0, c.delta)
    gp, gn = first_level_g(c.window(spike), c.delta)
    c.witness = {
        "single-plateau windows have one level": bool(np.all(nl[plateaus] == 1)),
        "plateau lengths around the table end": sorted((c.w1 - c.w0)[plateaus].tolist()) == [8207, 8208, 8209, 8217, 9000, 16384],
        "a step detected after the table end": nl[stepped] == 2 and ed[stepped, 1] == SEQ_TAB + 100,
        "spike increment at count SEQ_TAB is the definition's": s_tab[0] == sp[SEQ_TAB - 2],
        "the two reciprocals fall on either side of H": s_tab[0] != s_div[0] and int(np.rint(F32(c.h) * F32(1024))) == H,
        "statistics are 0 before the spike": gp[SEQ_TAB - 2] == 0 and gn[SEQ_TAB - 2] == 0,
        "the spike decides a detection": (nl[spike] >= 2) == (s_tab[0] > H),
    }
    return c


@functools.lru_cache(maxsize=None)
def quiet_sum(delta: float, h: float) -> Case:
    """Windows whose first sample is a spike far above a long plateau: the sum of the deviations from the anchor grows
    by the spike at every sample.  The lanes add a group's deviations in 32 bits while the sum is below 2^30 and take the
    64-bit path beyond.  delta = 400 (the issue's case): the sum passes 2^30 inside the table; delta = 1e5 widens the
    quiet band so far that a sum wrapped at 2^32 would still look quiet, so only the guard keeps it out."""
    T = _Trace(int(delta + h))
    spikes = (6000.0, 20000.0) if delta < 1e4 else (31250.0, 40000.0)
    rows = []
    for amp in spikes:
        for L in (9000, 12000, 16384):
            x = T.noise(L)
            x[0] += amp
            rows.append(T.segment(x))
    c = T.case(f"quiet_sum_d{delta:g}_h{h:g}", delta=delta, h=h, min_rows=LANES)
    hq = F32(F32(F32(delta) * F32(64.0)) * F32(0.5))
    cross30, wrapped_quiet = [], []
    for i in rows:
        Sd = quiet_sums(c.window(i))
        cross30.append(int(np.argmax(np.abs(Sd) >= 2 ** 30)) if np.any(np.abs(Sd) >= 2 ** 30) else -1)
        k = np.arange(1, min(Sd.size, SEQ_TAB - 8))
        d = (eo.cusum_quantise(c.window(i)) - eo.cusum_quantise(c.window(i))[0])[k]
        t = (d.astype(F32) - (wrap32(Sd[k]).astype(F32) * (F32(1.0) / (k + 1).astype(F32))).astype(F32)).astype(F32)
        wrapped_quiet.append(bool(np.any((wrap32(Sd[k]) != Sd[k]) & (np.abs(t) <= hq))))
    c.witness = {
        "one level per window": bool(np.all(twin(c)[0][rows] == 1)),
        "the quiet sum passes 2^30 inside the table": all(0 < k < SEQ_TAB - 8 for k in cross30),
    }
    if delta >= 1e4:
        c.witness["a sum wrapped at 2^32 passes the quiet test"] = all(wrapped_quiet)
    return c


@functools.lru_cache(maxsize=None)
def clamp(kind: str) -> Case:
    """Near-constant plateaus (two values 1/64 pA apart: a variance of a quarter unit) followed by a jump, so that an
    increment reaches the clamp SMAX.  kind 'step': a step of 1000 pA, larger than delta (h = 10).  kind 'spike': one
    sample delta = 400 pA high (the height that gives the largest increment), and h = SMAX / 1024: the clamped increment
    equals H and detects nothing, an unclamped one would detect the spike."""
    T = _Trace(11 if kind == "step" else 12)
    rows = []
    h = 10.0 if kind == "step" else SMAX / 1024.0
    plateaus = (5000, 6000, 9000, 12000) if kind == "spike" else (600, 5000, 9000, 12000)
    for L in plateaus:
        x = 5000.0 + (np.arange(L + 300) % 2) / 64.0
        if kind == "step":
            x[L:] -= 1000.0
        else:
            x[L] += 400.0
        rows.append(T.segment(x))
    c = T.case(f"clamp_{kind}", h=h, min_rows=LANES)
    nl = twin(c)[0]
    reach, over = [], []
    for i, L in zip(rows, plateaus):
        sp, sn = eo.cusum_increments(eo.cusum_quantise(c.window(i)), 0, c.delta)
        reach.append(bool(np.any(np.abs(np.concatenate((sp, sn))) == SMAX)))
        a, b = increment_at(c.window(i), L, c.delta, F32(1.0) / F32(L + 1), clamp=False)
        over.append(bool(max(abs(a), abs(b)) > SMAX + 200000))
    c.witness = {
        "an increment reaches the clamp": all(reach),
        "levels": bool(np.all(nl[rows] == (2 if kind == "step" else 1))),
    }
    if kind == "spike":
        c.witness["the unclamped increment at the spike is above H"] = all(over)
    return c


@functools.lru_cache(maxsize=None)
def _levels_trace() -> _Trace:
    T = _Trace(5)
    T.rows_special = []
    for L, period in ((41 * 25, 25), (42 * 25, 25), (71 * 25, 25), (300, 100), (3000, 500), (SEQ_MAX, 16), (20000, 16)):
        x = T.noise(L) + 900.0 * (np.arange(L) // period % 2)             # L / period - 1 jumps
        T.rows_special.append(T.segment(x))
    T.filler(LANES - len(T.rows))
    return T


@functools.lru_cache(maxsize=None)
def levels(max_levels: int) -> Case:
    """Windows of 40, 41, 70, 1023 and 1249 alternating jumps: the level table fills and overflows at every max_levels
    (the lanes then re-read the rest of the window as the last level); at 1024 the 16384-sample window of the lanes
    fills the table exactly and the 20000-sample window of the warps overflows it."""
    T = _levels_trace()
    c = T.case(f"levels_{max_levels}", max_levels=max_levels)
    nl, _, _, _, ovf = twin(c)
    rows = T.rows_special
    full = c_twin.cusum_batch(*flat(subset(c, rows)), c.delta, c.h, 1024)
    lanes_ovf = ovf[rows] & ((c.w1 - c.w0)[rows] <= SEQ_MAX)
    c.witness = {
        "every jump is detected": full[0].tolist() == [41, 42, 71, 3, 6, 1024, 1024] and full[4].tolist() == [0] * 6 + [1],
        "the table fills on the lanes (and overflows below 1024)": bool(lanes_ovf.any()) if max_levels < 1024 else nl[rows[5]] == 1024,
        "overflowing rows fill the table": bool(np.all(nl[ovf == 1] == max_levels)),
        "finalize takes the per-entry kernel" if 32 % max_levels == 0 else "finalize takes the per-event kernel": True,
    }
    return c


@functools.lru_cache(maxsize=None)
def domain() -> Case:
    """Signs and size: a -5000 pA baseline with upward events, a trace that crosses 0, jumps of +-1e5 pA (the domain is
    |x - x0| < 2^23 / 64 pA), and a constant window longer than the reciprocal table (variance 0: no information)."""
    T = _Trace(9)
    neg = [T.segment(T.steps(L, 2, depth=-1600.0, base=-5000.0)) for L in (400, 2500, 9000)]
    cross = T.noise(3000, base=300.0)
    cross[1000:2000] -= 800.0
    cross[2500:] -= 350.0
    zc = T.segment(cross)
    big = T.noise(10000, base=0.0)
    big[2000:4000] += 1e5; big[6000:8000] -= 1e5
    jumps = T.segment(big)
    ramp = T.segment(-30000.0 + 1e5 * (np.arange(900) >= 300) + 24 * T.rng.standard_normal(900))
    const = T.segment(np.full(9000, 1234.5))
    c = T.case("domain", min_rows=LANES)
    nl, ed = twin(c)[0], twin(c)[1]
    dmax = max(int(np.abs(eo.cusum_quantise(c.window(i))).max()) for i in (jumps, ramp))
    c.witness = {
        "negative baseline, upward events": bool(np.all(c.window(neg[0]) < 0)) and nl[neg[0]] == 3,
        "a window crossing 0": bool(c.window(zc).min() < 0 < c.window(zc).max()) and nl[zc] >= 3,
        "jumps of 1e5 pA inside the domain": 0.98e5 * 64 < dmax < 2 ** 23,
        "every 1e5 jump detected": nl[jumps] == 5 and nl[ramp] == 2,
        "constant window beyond the table has one level": nl[const] == 1 and c.w1[const] - c.w0[const] > SEQ_TAB,
    }
    return c


PARAMS = [(400.0, H_MAX), (400.0, 1.0 / 1024), (1e-3, 10.0), (1e5, 10.0)]


@functools.lru_cache(maxsize=None)
def params(delta: float, h: float) -> Case:
    """The accepted ends of the parameter range: h = 2^18 (H = 2^28), h = 1/1024 (H = 1), delta = 1e-3 (a quiet band of
    0.032 units: no sample is quiet) and delta = 1e5 (every sample of a noisy trace is quiet)."""
    T = _Trace(13)
    rows = [T.segment(T.steps(L, k)) for L, k in ((60, 1), (500, 3), (3000, 8), (9000, 4), (20000, 6))]
    rows.append(T.segment(T.noise(700)))
    c = T.case(f"params_d{delta:g}_h{h:g}", delta=delta, h=h, min_rows=LANES)
    nl, _, _, _, ovf = twin(c)
    H = int(np.rint(F32(h) * F32(1024)))
    w = {"H": H == {H_MAX: 2 ** 28, 1.0 / 1024: 1}.get(h, 10240)}
    if h == H_MAX or delta == 1e5:
        w["no window has a second level"] = bool(np.all(nl[rows] == 1))
    if h == 1.0 / 1024:
        x, offs = flat(c)
        w["H = 1 detects more than H = 10240"] = int(nl.sum()) > int(c_twin.cusum_batch(x, offs, delta, 10.0, c.max_levels)[0].sum())
    if delta in (1e-3, 1e5):
        qf = quiet_fraction(c.window(rows[-1]), delta)
        w["quiet samples on a plateau"] = qf < 0.01 if delta == 1e-3 else qf == 1.0
    c.witness = w
    return c


@functools.lru_cache(maxsize=None)
def rejected() -> Case:
    """Windows the kernels must reject, mixed into a batch the lanes take: empty, reversed, starting before 0, ending
    beyond the trace, longer than 2^30 samples, and accepted windows of types 2 and 3."""
    T = _Trace(17)
    good = [T.segment(T.steps(L, 2)) for L in (100, 2000)]
    bad = [T.window(50, 50), T.window(300, 200), T.window(-5, 40), T.window(-1, 0),
           T.segment(T.steps(200, 2), typ=2), T.segment(T.steps(200, 2), typ=3)]
    T.filler(LANES - len(T.rows) - 3)
    n = T.size + 5000
    bad += [T.window(n - 100, n + 1), T.window(0, MAX_WINDOW + 1), T.window(10, 10 + MAX_WINDOW + 1)]
    T.add(T.noise(5000))
    c = T.case("rejected")
    ok = accepted(c.y, c.w0, c.w1, c.types)
    c.witness = {
        "every kind of rejected window": not ok[bad].any() and ok[good].all() and c.y.size == n,
    }
    c.groups["bad"] = bad
    return c


CAPACITY = 40000
DEVICE_COUNTS = (0, 1, SEQ_MIN_EVENTS - 1, SEQ_MIN_EVENTS, 30000, CAPACITY)


@functools.lru_cache(maxsize=None)
def device_rows() -> Case:
    """CAPACITY rows of windows as the detector leaves them (short ones, long ones for the warps, rejected types);
    `device_batch` overwrites the rows at or beyond a device-side count with garbage."""
    T = _Trace(19)
    base = []
    for L in np.concatenate((T.rng.integers(20, 3000, 1200), [SEQ_MAX + 1, 17000, 20000])):
        base.append(T.segment(T.steps(int(L), int(T.rng.integers(0, 4))), typ=2 if T.rng.random() < 0.03 else 0))
    w = np.array(T.rows, np.int64)
    order = T.rng.permutation(CAPACITY) % len(base)
    order[-1] = base[0]                                        # the last row: an accepted window
    T.rows = [tuple(w[i]) for i in order]
    c = T.case("device_rows")
    lens = c.w1 - c.w0
    beyond = [~accepted(c.y, *_garbage(c, k))[k:] for k in DEVICE_COUNTS[:-1]]
    c.witness = {
        "long windows for the warps below the counts around SEQ_MIN_EVENTS": all(np.any(lens[:k] > SEQ_MAX) for k in DEVICE_COUNTS[2:]),
        "rejected types": bool(np.any(c.types != 0)),
        "rows beyond a count: garbage and stale accepted windows, the last one accepted": all(b.any() and (~b).any() and not b[-1] for b in beyond),
    }
    return c


def device_batch(count: int):
    """(w0, w1, types) of `device_rows` with rows at or beyond `count` replaced by stale and garbage windows: reversed,
    beyond the trace, longer than 2^30, type 2, and accepted windows of type 0 (left from an earlier run); the last row
    is always such an accepted window."""
    return _garbage(device_rows(), count)


def _garbage(c: Case, count: int):
    w0, w1, ty = c.w0.copy(), c.w1.copy(), c.types.copy()
    for i in range(count, CAPACITY):
        k = (i - count) % 5
        if i == CAPACITY - 1 or k == 4:
            continue                                          # a stale window of type 0 or 2 from an earlier run
        w0[i], w1[i], ty[i] = [(w1[i], w0[i], 0), (w0[i], c.y.size + 3, 0), (1, 2 + MAX_WINDOW, 0), (w0[i], w1[i], 2)][k]
    return w0, w1, ty


def _key(f, a) -> str:
    return "-".join([f.__name__] + [f"{v:g}" if isinstance(v, float) else str(v) for v in a])


# every builder with the arguments the tests use, by test id
BUILDERS = {_key(c, a): functools.partial(c, *a) for c, a in
            [(dispatch, (SEQ_MIN_EVENTS - 1,)), (dispatch, (SEQ_MIN_EVENTS,))] + [(line_grid, (t,)) for t in (0, 1, 13, 31)] +
            [(recip_table, ())] + [(quiet_sum, p) for p in ((400.0, 10.0), (400.0, 1000.0), (1e5, 10.0))] +
            [(clamp, ("step",)), (clamp, ("spike",))] + [(levels, (m,)) for m in (2, 3, 4, 32, 33, 64, 1024)] +
            [(domain, ())] + [(params, p) for p in PARAMS] + [(rejected, ()), (device_rows, ())]}
