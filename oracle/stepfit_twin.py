"""TEST INFRASTRUCTURE — float64 restatement of the step-fit kernel's own Levenberg-Marquardt loop.

`stepfit_oracle.py` stays the definition of the fit (scipy's MINPACK LM); it takes another path through the same cost
surface, so it can only be compared with the kernel by rates.  This module follows `ct_stepfit_kernel`
(cusumtools_b200/csrc/ct_stepfit.cu) decision for decision, with float64 where the kernel uses float32 sums:

  * the window relative to its first sample (a float32 subtraction, as the kernel stages it) and the initial guess
    i0 = mean of the 2 padding baseline samples, a = i0 - mean of the interior, u1 = padding, u2 = n - padding,
    tau1 = tau2 = tau0 rounded to float32 (the kernel's argument type);
  * floor_ = n (5.96e-8 max|x - x0|)^2, the float32 resolution of the cost;
  * the step solves (A + mu diag A) d = J^T r on the Jacobi-scaled matrix (unit diagonal) by Cholesky; mu0 = 1e-3,
    x10 after a rejected trial, x0.1 after an accepted one; a matrix that is not positive definite gives mu x10 and
    one more trial on the counter, without an evaluation;
  * stops: predicted decrease 2 d.g - d^T A d <= 1e-9 c + floor_, relative step < 1e-8 (the i0 denominator is the
    absolute level |p0 + x0|), and after an accepted trial an actual decrease < 1e-9 c + floor_;
  * a trial outside the domain (tau <= 0 or u1 >= u2) is not evaluated and still counts;
  * acceptance ct < c; loop guard it < max_iters and mu < 1e30; the validity rule and level rows of the kernel.

Every decision is recorded with its margin, the distance from its threshold in the units the kernel's float32 sums
blur: a GPU comparison can then skip the events where the kernel and the twin may decide a float32 tie differently.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field

import numpy as np

NPARAM = 6
MU0 = 1e-3
FLOAT32_RES = 5.96e-8          # 2^-24 as the kernel writes it


def window(x) -> tuple[np.ndarray, float]:
    """(x - x[0] as the kernel stages it: a float32 subtraction, widened to float64; x[0] as float32 -> float64)."""
    xf = np.asarray(x, np.float32)
    x0 = xf[0]
    return (xf - x0).astype(np.float64), float(x0)


def initial_point(xr: np.ndarray, padding: int, tau0: float) -> np.ndarray:
    """The kernel's initial guess in the window frame (i0 relative to x[0])."""
    n, P = xr.size, int(padding)
    i0 = float(np.concatenate((xr[:P], xr[n - P:])).sum()) / (2.0 * P)
    a = i0 - float(xr[P:n - P].sum()) / float(n - 2 * P)
    tau = float(np.float32(tau0))
    return np.array([i0, a, float(P), float(n - P), tau, tau])


def residual_and_jacobian(xr: np.ndarray, p) -> tuple[np.ndarray, np.ndarray]:
    """r = x - f and J = df/dp over the window, H(s) = [s >= 0] (H(0) = 1: the exponential starts at its sample)."""
    i0, a, u1, u2, t1, t2 = (float(v) for v in p)
    t = np.arange(xr.size, dtype=np.float64)
    s1, s2 = t - u1, t - u2
    h1, h2 = s1 >= 0, s2 >= 0
    with np.errstate(over="ignore"):
        e1 = np.where(h1, np.exp(-np.maximum(s1, 0.0) / t1), 0.0)
        e2 = np.where(h2, np.exp(-np.maximum(s2, 0.0) / t2), 0.0)
    dq = np.where(h2, 1.0 - e2, 0.0) - np.where(h1, 1.0 - e1, 0.0)
    J = np.empty((xr.size, NPARAM))
    J[:, 0] = 1.0
    J[:, 1] = dq
    J[:, 2] = a * e1 / t1
    J[:, 3] = -(a * e2 / t2)
    J[:, 4] = J[:, 2] * (s1 / t1)
    J[:, 5] = J[:, 3] * (s2 / t2)
    return xr - (i0 + a * dq), J


def sums(xr: np.ndarray, p) -> tuple[float, np.ndarray, np.ndarray]:
    """What one kernel pass leaves: (cost = sum r^2, g = J^T r [6], A = J^T J [6, 6])."""
    r, J = residual_and_jacobian(xr, p)
    return float(r @ r), J.T @ r, J.T @ J


def lm_step(g: np.ndarray, A: np.ndarray, mu: float):
    """(ok, d, predicted decrease, smallest Cholesky pivot of the scaled matrix).  ok is False (no step) when a
    diagonal entry of A is not positive or the scaled matrix is not positive definite."""
    diag = np.diag(A)
    if not np.all(diag > 0.0):
        return False, None, 0.0, math.inf
    sc = 1.0 / np.sqrt(diag)
    M = A * sc[:, None] * sc[None, :]
    np.fill_diagonal(M, 1.0 + mu)
    R = np.zeros((NPARAM, NPARAM))
    piv = math.inf
    for i in range(NPARAM):
        dii = M[i, i] - R[:i, i] @ R[:i, i]
        piv = min(piv, dii)
        if not dii > 0.0:
            return False, None, 0.0, piv
        R[i, i] = math.sqrt(dii)
        for j in range(i + 1, NPARAM):
            R[i, j] = (M[i, j] - R[:i, i] @ R[:i, j]) / R[i, i]
    b = g * sc
    z = np.zeros(NPARAM)
    for i in range(NPARAM):                      # R^T z = b
        z[i] = (b[i] - R[:i, i] @ z[:i]) / R[i, i]
    d = np.zeros(NPARAM)
    for i in reversed(range(NPARAM)):            # R d' = z
        d[i] = (z[i] - R[i, i + 1:] @ d[i + 1:]) / R[i, i]
    d *= sc
    return True, d, float(2.0 * (d @ g) - d @ A @ d), piv


def _rel(v: float, thr: float) -> float:
    m = max(abs(v), abs(thr))
    return abs(v - thr) / m if m > 0 else math.inf


@dataclass
class Step:
    """One pass of the loop; d is None where no step was solved."""
    kind: str                  # "no_pd", "stop_pred", "stop_rel", "domain", "accept", "reject"
    d: np.ndarray | None = None


@dataclass
class TwinFit:
    params: np.ndarray         # (i0 pA absolute, a, u1, u2, tau1, tau2), as the kernel reports them
    cost: float                # float64 sum of squared residuals at params
    iters: int
    type: int                  # 1 valid, 7 failed
    converged: bool
    initial: np.ndarray        # the initial guess, absolute i0
    steps: list[Step] = field(default_factory=list)
    margins: list[tuple[str, float]] = field(default_factory=list)   # (decision, distance from its threshold)
    edges: np.ndarray | None = None      # level rows of a valid fit: [0, ceil u1, ceil u2, n]
    mean: np.ndarray | None = None       # [i0, i0 - a, i0]
    std: np.ndarray | None = None        # rms of x - f over each level


def fit(x, padding: int, tau0: float, max_iters: int = 50) -> TwinFit:
    """The kernel's loop on one window x (the float32 samples of [win_start, win_end)).

    Margins: "pd" the smallest pivot of the unit-diagonal matrix; "pred" |pred - thr| / max(pred, thr); "rel"
    |big - 1e-8| / max(big, 1e-8); "domain" the smallest of tau_k and u2 - u1 of the trial relative to its size;
    "accept" |ct - c| / c; "decrease" |(c - ct) - thr| / c (thr = 1e-9 c + floor_); "valid" how far u1, u2 are from
    an integer (the ceil of the level edges), and tau from 0.05 and n, relative."""
    xr, x0 = window(x)
    n, P = xr.size, int(padding)
    if not 2 * P < n:
        raise ValueError("the window needs more than 2 padding samples")
    xs = float(np.abs(xr).max())
    floor_ = n * (xs * FLOAT32_RES) ** 2
    p = initial_point(xr, P, tau0)
    base_abs = x0 + p[0]
    init = p.copy()
    init[0] += x0
    c, g, A = sums(xr, p)
    it, mu, converged = 1, MU0, False
    steps, margins = [], []
    while it < max_iters and mu < 1e30:
        ok, d, pred, piv = lm_step(g, A, mu)
        margins.append(("pd", abs(piv)))
        if not ok:
            mu *= 10.0
            it += 1
            steps.append(Step("no_pd"))
            continue
        thr = 1e-9 * c + floor_
        margins.append(("pred", _rel(pred, thr)))
        if not pred > thr:
            converged = True
            steps.append(Step("stop_pred", d))
            break
        den = np.abs(p) + 1e-8
        den[0] = abs(p[0] + x0) + 1e-8
        big = float(np.max(np.abs(d) / den))
        margins.append(("rel", _rel(big, 1e-8)))
        if big < 1e-8:
            converged = True
            steps.append(Step("stop_rel", d))
            break
        q = p + d
        margins.append(("domain", min(abs(q[4]) / (abs(p[4]) + abs(d[4])), abs(q[5]) / (abs(p[5]) + abs(d[5])),
                                      abs(q[3] - q[2]) / (abs(p[3] - p[2]) + abs(d[3] - d[2])))))
        if not (q[4] > 0.0 and q[5] > 0.0 and q[2] < q[3]):
            mu *= 10.0
            it += 1
            steps.append(Step("domain", d))
            continue
        ct, gt, At = sums(xr, q)
        it += 1
        margins.append(("accept", abs(ct - c) / c if c > 0 else math.inf))
        if ct < c:
            steps.append(Step("accept", d))
            margins.append(("decrease", abs((c - ct) - thr) / c))
            dec = c - ct
            p, c, g, A = q, ct, gt, At
            mu *= 0.1
            if dec < thr:
                converged = True
                break
        else:
            steps.append(Step("reject", d))
            mu *= 10.0
    e1, e2 = math.ceil(p[2]), math.ceil(p[3])
    sign_ok = p[1] > 0.0 if base_abs >= 0.0 else p[1] < 0.0
    valid = (converged and p[2] > 0.0 and e1 < e2 and e2 < n and 0.05 <= p[4] <= n and 0.05 <= p[5] <= n and sign_ok)
    fr = [abs(u - round(u)) for u in (p[2], p[3])]
    margins.append(("valid", min(fr + [_rel(p[4], 0.05), _rel(p[4], n), _rel(p[5], 0.05), _rel(p[5], n)])))
    out = p.copy()
    out[0] += x0
    res = TwinFit(out, c, it, 1 if valid else 7, converged, init, steps, margins)
    if valid:
        r, _ = residual_and_jacobian(xr, p)
        res.edges = np.array([0, e1, e2, n], np.int64)
        res.mean = np.array([out[0], out[0] - out[1], out[0]])
        res.std = np.array([math.sqrt(np.mean(r[lo:hi] ** 2)) for lo, hi in ((0, e1), (e1, e2), (e2, n))])
    return res


def cost_at(x, params) -> float:
    """float64 sum of squared residuals of the window x at a reported parameter row (absolute i0)."""
    x = np.asarray(x, np.float64)
    r, _ = residual_and_jacobian(x, params)
    return float(r @ r)


def filtered_pulse_windows(sizes, padding: int, seed: int, noise: float = 150.0, samplerate: float = 4166666.0,
                           cutoff: float = 1e5, order: int = 8) -> list[np.ndarray]:
    """One float32 window per entry of `sizes` (samples): a rectangular pulse of size - 2 padding samples, depth
    uniform in 300-2000 pA toward zero from a baseline of +5000 pA (even entries) or -5000 pA (odd ones), in white
    noise of `noise` pA, through the reference's filter (scipy bessel + filtfilt) with 400 samples of baseline either
    side of the window."""
    from scipy import signal
    rng = np.random.default_rng(seed)
    b, a = signal.bessel(int(order), 2.0 * cutoff / samplerate)
    guard = 400
    out = []
    for k, n in enumerate(sizes):
        sgn = 1.0 if k % 2 == 0 else -1.0
        x = np.full(int(n) + 2 * guard, sgn * 5000.0)
        x[guard + padding:guard + int(n) - padding] -= sgn * rng.uniform(300.0, 2000.0)
        x += noise * rng.standard_normal(x.size)
        out.append(signal.filtfilt(b, a, x)[guard:guard + int(n)].astype(np.float32))
    return out


def local_minimum_gap(x, params) -> tuple[float, float]:
    """Certificate of a fit: scipy's float64 LM (stepfit_oracle's residuals and domain), started at `params`.
    Returns (relative cost decrease it finds, largest parameter move in standard errors at `params`)."""
    from scipy.optimize import least_squares

    from . import stepfit_oracle as so
    x = np.asarray(x, np.float64)
    n = x.size
    c0 = cost_at(x, params)
    big = np.full(n, 1e12)
    r = least_squares(lambda p: so.model(p, n) - x if so.in_domain(p) else big, np.asarray(params, np.float64),
                      jac=lambda p: so.jacobian(p, n) if so.in_domain(p) else np.zeros((n, NPARAM)), method="lm",
                      xtol=1e-14, ftol=1e-14, gtol=1e-14, max_nfev=2000)
    c1 = cost_at(x, r.x)
    se = so.standard_errors(x, params)
    return max(0.0, (c0 - c1) / c0), float(np.max(np.abs(r.x - params) / se))
