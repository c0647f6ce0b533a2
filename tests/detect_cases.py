"""Traces that drive the event detector (csrc/ct_detect.cu) across every boundary of its scan, built from a segment list
with an exact reference, at any length up to and past 2^32 samples.

A case is a list of segments (start, class) over n samples and one pair of lines per baseline block.  The class of a
segment is the symbol every one of its samples has against its block's lines:
  A  beyond the start line;
  N  no symbol: strictly between the lines, exactly on the start line or exactly on the end line;
  B  back beyond the end line.
`materialise` turns the list into the float32 trace, in chunks, on any torch device: a sample's value is made in the
mirrored frame (v' = sign * v, where "beyond" is always "below") - A: ts' - 1 - 40u, B: te' + 1 + 40u, N: ts', te' or a
value strictly between them - and y = sign * v' (the sign flip is exact).  `reference` runs the detector's automaton over
the segments, O(segments), so it is exact at any length: a start is the first A after outside, an end the first B
after inside.

The lines respect the detector's precondition, sign * t_start <= sign * t_end per block (ts' == te' included).

The scan the cases aim at (ct_detect_f32): runs of RUN samples (one warp each in pass 1), groups of GROUP runs (one
thread each in ct_detect_scan_groups), and the single-CTA scan where each of 1024 threads owns per = ceil(ng / 1024)
consecutive groups.  Every builder returns a witness, named facts computed from the segment list that show the case
reaches what it is named for.  tests/test_detect_cases_host.py checks the reference against the three forms of the
definition and every witness; tests/test_gpu_detect_scale.py runs the kernels on the same cases.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np
import torch

RUN = 4096                      # kRun: samples per pass-1 warp run
GROUP = 64                      # kGroup: runs per group of the scan
GROUP_SAMPLES = RUN * GROUP     # 2^18
SCAN_THREADS = 1024             # threads of the single-CTA scan
N_, A_, B_ = 0, 1, 2            # segment classes
C2_SAMPLES = 2_499_999_600      # samples of one benchmark step (bench.py, config C2)
CHUNK = 1 << 26                 # samples materialised per step


@dataclass(eq=False)
class Case:
    name: str
    n: int
    block: int
    sign: np.ndarray            # int32 [nb]
    t_start: np.ndarray         # float32 [nb]
    t_end: np.ndarray           # float32 [nb]
    seg_start: np.ndarray       # int64, strictly increasing, seg_start[0] == 0, all < n
    seg_class: np.ndarray       # int8 (N_, A_, B_)
    state_in: bool = False
    witness: dict = field(default_factory=dict)

    @property
    def nruns(self) -> int:
        return -(-self.n // RUN)

    @property
    def ng(self) -> int:
        return -(-self.nruns // GROUP)

    @property
    def per(self) -> int:
        return -(-self.ng // SCAN_THREADS)

    @property
    def range_samples(self) -> int:
        """Samples of one thread range of the single-CTA scan."""
        return self.per * GROUP_SAMPLES


def scan_shape(n: int):
    """(nruns, ng, per) of ct_detect_f32 on n samples."""
    nruns = -(-n // RUN)
    ng = -(-nruns // GROUP)
    return nruns, ng, -(-ng // SCAN_THREADS)


def lines(nb: int, seed: int, hysteresis=(0.0, 1.0, 2.5)):
    """Per-block sign and float32 lines: baselines of both signs, and end lines on, near and away from the start line."""
    rng = np.random.default_rng(seed)
    sign = np.where(rng.random(nb) < 0.5, 1, -1).astype(np.int32)
    mean = sign * (5000.0 + rng.integers(0, 300, nb))
    std = 10.0 + rng.integers(0, 20, nb)
    hyst = np.asarray(hysteresis, np.float64)[rng.integers(0, len(hysteresis), nb)]
    t_start = (mean - sign * 5.0 * std).astype(np.float32)
    t_end = (mean - sign * (5.0 - hyst) * std).astype(np.float32)
    return sign, t_start, t_end


# ---------------------------------------------------------------------------------------------------------- reference
def reference_raw(c: Case):
    """Every start and every end the automaton produces, in time order, as the kernel's counters count them: with
    state_in the first end may close an event opened before the data, and the last start may still be open."""
    ss, cc = c.seg_start, c.seg_class
    starts, ends = [], []
    inside = bool(c.state_in)
    for p, k in zip(ss.tolist(), cc.tolist()):
        if k == A_ and not inside:
            inside = True
            starts.append(p)
        elif k == B_ and inside:
            inside = False
            ends.append(p)
    return np.array(starts, np.int64), np.array(ends, np.int64)


def events_form(starts, ends, state_in: bool):
    """Raw lists -> (starts, ends, open_start), the form of eo.detect_events and detect.detect_events."""
    if state_in and ends.size and (starts.size == 0 or ends[0] < starts[0]):
        ends = ends[1:]
    open_start = -1
    if starts.size > ends.size:
        open_start = int(starts[-1])
        starts = starts[:-1]
    return starts, ends, open_start


def reference(c: Case):
    return events_form(*reference_raw(c), c.state_in)


# -------------------------------------------------------------------------------------------------------- the trace
def materialise(c: Case, device, out: torch.Tensor | None = None, seed: int = 0, chunk: int = CHUNK) -> torch.Tensor:
    """The float32 trace of `c` on `device`, generated chunk by chunk (the same code at every size)."""
    y = torch.empty(c.n, dtype=torch.float32, device=device) if out is None else out
    ss = torch.from_numpy(c.seg_start).to(device)
    cls = torch.from_numpy(c.seg_class.astype(np.int64)).to(device)
    sg = torch.from_numpy(c.sign.astype(np.float32)).to(device)
    ts = sg * torch.from_numpy(c.t_start).to(device)              # mirrored lines, exact
    te = sg * torch.from_numpy(c.t_end).to(device)
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    for c0 in range(0, c.n, chunk):
        c1 = min(c.n, c0 + chunk)
        idx = torch.arange(c0, c1, device=device, dtype=torch.int64)
        k = cls[torch.searchsorted(ss, idx, right=True) - 1]
        kb = idx // c.block
        del idx
        a, b, s = ts[kb], te[kb], sg[kb]
        del kb
        u = torch.rand(c1 - c0, generator=g, device=device, dtype=torch.float32)
        mid = a + (b - a) * u
        # N: on the start line, on the end line, or strictly between them (when they differ)
        vn = torch.where(u < 0.25, a, torch.where(u < 0.5, b, torch.where((mid > a) & (mid < b), mid, a)))
        v = torch.where(k == A_, a - 1.0 - 40.0 * u, torch.where(k == B_, b + 1.0 + 40.0 * u, vn))
        y[c0:c1] = s * v
        del k, a, b, s, u, mid, vn, v
    return y


def symbols_match(c: Case, y: torch.Tensor, chunk: int = CHUNK) -> bool:
    """Every sample's symbol against its block's lines is its segment's class (plain torch comparisons, no kernel)."""
    dev = y.device
    ss = torch.from_numpy(c.seg_start).to(dev)
    cls = torch.from_numpy(c.seg_class.astype(np.int64)).to(dev)
    sg = torch.from_numpy(c.sign.astype(np.float32)).to(dev)
    ts = sg * torch.from_numpy(c.t_start).to(dev)
    te = sg * torch.from_numpy(c.t_end).to(dev)
    ok = True
    for c0 in range(0, c.n, chunk):
        c1 = min(c.n, c0 + chunk)
        idx = torch.arange(c0, c1, device=dev, dtype=torch.int64)
        k = cls[torch.searchsorted(ss, idx, right=True) - 1]
        kb = idx // c.block
        v = sg[kb] * y[c0:c1]
        sym = torch.where(v < ts[kb], A_, torch.where(v > te[kb], B_, N_))
        ok = ok and bool((sym == k).all())
    return ok


# ------------------------------------------------------------------------------------------------------- builders
# Each pattern puts a few segments around a point p (all inside [p - 8, p + 12)) and leaves the state outside.
PATTERNS = {
    "start": ((-6, B_), (-3, N_), (0, A_), (4, N_), (8, B_), (11, N_)),      # an event starts at p
    "end": ((-8, A_), (-4, N_), (0, B_), (2, N_)),                          # an event ends at p
    "inner": ((-5, A_), (-2, N_), (0, A_), (3, B_), (6, N_)),               # a class change at p inside an event
    "across": ((-8, B_), (-5, A_), (-2, N_), (3, B_), (6, N_)),             # an event spans p, no symbol at p
}
ORDER = ("start", "end", "inner", "across")
SPAN = (-8, 12)


def _pattern_facts(p: int, kind: str, starts, ends, seg):
    if kind == "start":
        return p in starts
    if kind == "end":
        return p in ends
    if kind == "inner":
        return p in seg and p not in starts and p not in ends
    i = np.searchsorted(starts, p, side="right") - 1                    # across: the last start before p ends after p
    return i >= 0 and i < ends.size and ends[i] > p and p not in seg


def layout(name: str, n: int, block: int, state_in: bool, points: dict, *, rot: int = 0, seed: int = 0,
           long_inside: int | None = None, quiet_outside: int | None = None, open_last: bool = True) -> Case:
    """A case from named point lists: points[category] = exact sample positions (run, group or scan-range boundaries,
    2^31 ...).  The patterns start / end / inner / across go to the points of each category in turn (rotated by `rot`).
    `long_inside` = t: an event from just before scan range t to just after range t + 1, so one whole thread range
    lies inside it with no symbol; `quiet_outside` = t: the same stretch with no symbol, outside any event.
    `open_last`: an event starts on the last sample and is still open at the end."""
    rs = scan_shape(n)[2] * GROUP_SAMPLES
    segs = {0: N_}
    busy = []                                                            # [a, b) spans that patterns must avoid
    for t, first, last in ((long_inside, A_, B_), (quiet_outside, B_, A_)):
        if t is None:
            continue
        a, b = t * rs - 5, (t + 2) * rs + 7
        assert 8 <= a and b + 16 <= n
        segs[a], segs[a + 1], segs[b] = first, N_, last
        segs[b + 4], segs[b + 8], segs[b + 11] = N_, B_, N_              # back outside after a quiet stretch's event
        busy.append((a - 8, b + 12))
    if open_last:
        segs[n - 5], segs[n - 4], segs[n - 1] = B_, N_, A_
        busy.append((n - 5, n))
    placed = []
    taken = set()
    for cat, pts in points.items():
        for j, p in enumerate(pts):
            kind = ORDER[(j + rot) % len(ORDER)]
            lo, hi = p + SPAN[0], p + SPAN[1]
            if lo < 1 or hi > n or p in taken or any(lo < b and a < hi for a, b in busy):
                continue
            for d, k in PATTERNS[kind]:
                segs[p + d] = k
            busy.append((lo, hi))
            taken.add(p)
            placed.append((cat, p, kind))
    pos = np.array(sorted(segs), np.int64)
    c = Case(name, n, block, *lines(-(-n // block), seed), pos, np.array([segs[p] for p in pos.tolist()], np.int8),
             state_in)
    starts, ends = reference_raw(c)
    ev_s, ev_e, _ = events_form(starts, ends, state_in)       # paired: event i is [ev_s[i], ev_e[i])
    seg = set(c.seg_start.tolist())
    sset, eset = set(starts.tolist()), set(ends.tolist())
    w = c.witness
    for cat, p, kind in placed:
        w[f"{kind}_on_{cat}@{p}"] = _pattern_facts(p, kind, sset if kind != "across" else ev_s,
                                                   eset if kind != "across" else ev_e, seg)
    for cat in points:
        w[f"some_pattern_on_{cat}"] = any(q[0] == cat for q in placed)
    if long_inside is not None:
        t = long_inside
        a, b = t * rs - 5, (t + 2) * rs + 7
        i = np.searchsorted(ev_s, a)
        w["long_event_covers_a_whole_scan_range"] = (i < ev_s.size and ev_s[i] == a and i < ev_e.size
                                                     and ev_e[i] == b and b - a > 2 * rs)
        w["long_event_range_has_no_symbol"] = not np.any((c.seg_start > a + 1) & (c.seg_start < b))
    if quiet_outside is not None:
        t = quiet_outside
        a, b = t * rs - 5, (t + 2) * rs + 7
        w["quiet_range_is_outside"] = _outside_at(starts, ends, a, c.state_in)
        w["quiet_range_has_no_symbol"] = not np.any((c.seg_start > a + 1) & (c.seg_start < b))
        w["quiet_range_ends_with_a_start"] = b in sset
    if open_last:
        w["open_event_starts_on_the_last_sample"] = events_form(starts, ends, state_in)[2] == n - 1
    return c


def _outside_at(starts, ends, p, state_in):
    """True if the automaton is outside at sample p (after p's own symbol)."""
    ns = np.searchsorted(starts, p, side="right")
    ne = np.searchsorted(ends, p, side="right")
    return ns + int(state_in) <= ne


def boundary_points(n: int, block: int, extra: dict | None = None) -> dict:
    """Points on the run, group, scan-range and block boundaries of an n-sample trace, and one sample either side of
    some of them (the last sample of one piece and the first of the next)."""
    nruns, ng, per = scan_shape(n)
    rs = per * GROUP_SAMPLES
    nr = -(-n // rs)
    pts = {
        "run": [RUN * k for k in (3, 70, 1001, 4099, nruns - 70) if 0 < RUN * k < n and (RUN * k) % GROUP_SAMPLES],
        "group": [GROUP_SAMPLES * k for k in (1, 2, 5, 7, ng - 2) if 0 < GROUP_SAMPLES * k < n
                  and (GROUP_SAMPLES * k) % rs],
        "range": [rs * t for t in (1, 2, 3, nr // 3, nr - 2, nr - 1) if 0 < rs * t < n],
        "range_minus_1": [rs * t - 1 for t in (4, nr // 3 + 1) if 0 < rs * t - 1 < n],
        "range_plus_1": [rs * t + 1 for t in (5, nr // 3 + 2) if 0 < rs * t + 1 < n],
        "block": [block * k for k in (1, 3, 6, 11, -(-n // block) - 1) if 0 < block * k < n],
    }
    pts.update(extra or {})
    return {k: sorted(set(v)) for k, v in pts.items() if v}


def scale_case(n: int, block: int, state_in: bool, variant: int = 0, extra: dict | None = None) -> Case:
    """A trace of n samples with patterns on every boundary kind, one long event over a whole scan range, one quiet
    range outside any event and an open event on the last sample."""
    nr = -(-n // (scan_shape(n)[2] * GROUP_SAMPLES))
    return layout(f"n{n}_b{block}_s{int(state_in)}", n, block, state_in, boundary_points(n, block, extra), rot=variant,
                  seed=variant + 17 * int(state_in) + block % 977, long_inside=nr // 2, quiet_outside=nr // 2 + 4)


def big_points(n: int) -> dict:
    """2^31 and 2^32 (when inside the trace) and run boundaries around them."""
    out = {}
    for e in (31, 32):
        p = 1 << e
        if p + 64 * RUN < n:
            out[f"2^{e}"] = [p]
            out[f"runs_near_2^{e}"] = [p - 7 * RUN, p + 3 * RUN, p + 9 * RUN, p + 40 * RUN]
    return out


SCAN_SIZES = (1 << 28, (1 << 28) + 1, (1 << 29) + 1)
BIG_SIZES = (C2_SAMPLES, (1 << 32) + (1 << 20) + 13)
BLOCKS = (4096, 1 << 20)


def scan_cases(n: int):
    """The four variants (block, state_in) of an n-sample case, patterns rotated so that over them every boundary kind
    sees every pattern."""
    extra = big_points(n)
    return [scale_case(n, b, s, variant=2 * i + int(s), extra=extra) for i, b in enumerate(BLOCKS) for s in (False, True)]


def small_case(n: int, block: int, state_in: bool, seed: int) -> Case:
    """A random segment list over a short trace (host tests): segments of 1 to 300 samples, random classes."""
    rng = np.random.default_rng(seed)
    cuts = [0]
    while True:
        nxt = cuts[-1] + int(rng.integers(1, 300))
        if nxt >= n:
            break
        cuts.append(nxt)
    cls = rng.choice(np.array([N_, A_, B_], np.int8), len(cuts), p=[0.4, 0.3, 0.3])
    return Case(f"small_n{n}_b{block}_s{int(state_in)}_{seed}", n, block, *lines(-(-n // block), seed),
                np.array(cuts, np.int64), cls, state_in)
