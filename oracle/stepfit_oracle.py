"""TEST INFRASTRUCTURE — NumPy/SciPy DEFINITION of the step-response fit of short events (rate.csv type 1).

The reference repo has no implementation of this fit: it only consumes its result (`readevents.py:1334-1337` reads a
type-1 event file with the columns time, current, cusum, stepfit; `plot-trace.py:354-357` counts types 0 and 1 as
good events; events.csv has `rc_const1_us` / `rc_const2_us`).  The model is the step response the upstream event
fitter uses for short events (two exponential edges, one amplitude, two RC time constants; SURVEY.md Appendix C, from
recalled knowledge, not reference code), so this module IS the definition, as events_oracle.py is for CUSUM+.

For window sample t = 0 .. n-1 and p = (i0, a, u1, u2, tau1, tau2) (pA, pA, samples x 4):
    f(t) = i0 - a (1 - exp(-(t-u1)/tau1)) H(t-u1) + a (1 - exp(-(t-u2)/tau2)) H(t-u2),   H(s) = [s >= 0]
Initial guess (`initial_guess`, shared with the kernel), validity (`is_valid`), level rows (`level_rows`) and the
parameter standard errors (`standard_errors`) follow; `fit_event` minimises sum (x - f)^2 with
scipy.optimize.least_squares(method='lm') and the analytic Jacobian.  cost = sum of squared residuals (pA^2).
"""
from __future__ import annotations

import math

import numpy as np
from scipy.optimize import least_squares

NPARAM = 6
TAU_MIN = 0.05


def model(p, n: int) -> np.ndarray:
    i0, a, u1, u2, t1, t2 = (float(v) for v in p)
    t = np.arange(int(n), dtype=np.float64)
    s1, s2 = t - u1, t - u2
    e1 = np.where(s1 >= 0, np.exp(-np.maximum(s1, 0.0) / t1), 0.0)
    e2 = np.where(s2 >= 0, np.exp(-np.maximum(s2, 0.0) / t2), 0.0)
    q1 = np.where(s1 >= 0, 1.0 - e1, 0.0)
    q2 = np.where(s2 >= 0, 1.0 - e2, 0.0)
    return i0 - a * q1 + a * q2


def jacobian(p, n: int) -> np.ndarray:
    """df/dp, [n, 6] (the kink of H at t = u contributes nothing: 1 - exp(0) = 0)."""
    i0, a, u1, u2, t1, t2 = (float(v) for v in p)
    t = np.arange(int(n), dtype=np.float64)
    s1, s2 = t - u1, t - u2
    h1, h2 = s1 >= 0, s2 >= 0
    e1 = np.where(h1, np.exp(-np.maximum(s1, 0.0) / t1), 0.0)
    e2 = np.where(h2, np.exp(-np.maximum(s2, 0.0) / t2), 0.0)
    J = np.empty((t.size, NPARAM))
    J[:, 0] = 1.0
    J[:, 1] = np.where(h2, 1.0 - e2, 0.0) - np.where(h1, 1.0 - e1, 0.0)
    J[:, 2] = a * e1 / t1
    J[:, 3] = -a * e2 / t2
    J[:, 4] = a * e1 * s1 / (t1 * t1)
    J[:, 5] = -a * e2 * s2 / (t2 * t2)
    return J


def initial_guess(x, padding: int, tau0: float) -> np.ndarray:
    """i0 = mean of the first and last `padding` samples, a = i0 - mean of the rest, u1 = padding,
    u2 = n - padding, tau1 = tau2 = tau0."""
    x = np.asarray(x, np.float64)
    n, P = x.size, int(padding)
    i0 = float(np.concatenate((x[:P], x[n - P:])).mean())
    a = i0 - float(x[P:n - P].mean())
    return np.array([i0, a, float(P), float(n - P), float(tau0), float(tau0)])


def in_domain(p) -> bool:
    """Trial points outside it (tau <= 0 or u1 >= u2) are rejected without being evaluated."""
    return p[4] > 0 and p[5] > 0 and p[2] < p[3]


def fit_event(x, padding: int, tau0: float, max_nfev: int = 2000):
    """Least-squares fit of one window.  Returns (p float64[6], cost = sum (x - f)^2, converged, evaluations)."""
    x = np.asarray(x, np.float64)
    n = x.size
    x0 = float(x[0])
    xr = x - x0                                      # the window relative to its first sample, as the kernel sees it
    p0 = initial_guess(xr, padding, tau0)
    big = np.full(n, 1e12)

    def res(p):
        return model(p, n) - xr if in_domain(p) else big

    def jac(p):
        return jacobian(p, n) if in_domain(p) else np.zeros((n, NPARAM))

    r = least_squares(res, p0, jac=jac, method="lm", xtol=1e-14, ftol=1e-14, gtol=1e-14, max_nfev=max_nfev)
    p = r.x.copy()
    p[0] += x0
    cost = float(np.sum((model(p, n) - x) ** 2))
    return p, cost, bool(r.status > 0) and in_domain(r.x), int(r.nfev)


def is_valid(p, n: int, converged: bool, baseline: float) -> bool:
    """A fit is valid when it converged, every level row holds a sample (0 < u1, ceil u1 < ceil u2 < n, which gives
    0 < u1 < u2 < n), 0.05 <= tau1, tau2 <= n, and a has the sign of the blockage the detector saw: the current moves
    from the baseline toward zero (plot-trace.py:408-411), i.e. sign(a) = sign(baseline) with `baseline` the
    initial i0 (sign(0) = +1)."""
    i0, a, u1, u2, t1, t2 = (float(v) for v in p)
    if not converged or not (u1 > 0) or not (math.ceil(u1) < math.ceil(u2) < n):
        return False
    if not (TAU_MIN <= t1 <= n and TAU_MIN <= t2 <= n):
        return False
    return a > 0 if baseline >= 0 else a < 0


def level_rows(x, p):
    """(edges int64[4], mean float64[3], std float64[3]) of a valid fit: edges = [0, ceil u1, ceil u2, n],
    mean = [i0, i0 - a, i0], std = rms of x - f over each level."""
    x = np.asarray(x, np.float64)
    n = x.size
    e = np.array([0, math.ceil(p[2]), math.ceil(p[3]), n], np.int64)
    r = x - model(p, n)
    std = np.array([math.sqrt(np.mean(r[e[k]:e[k + 1]] ** 2)) for k in range(3)])
    return e, np.array([p[0], p[0] - p[1], p[0]]), std


def standard_errors(x, p) -> np.ndarray:
    """se_k = sqrt(diag((J^T J)^-1) * cost / (n - 6)) at p."""
    x = np.asarray(x, np.float64)
    n = x.size
    J = jacobian(p, n)
    cost = float(np.sum((x - model(p, n)) ** 2))
    return np.sqrt(np.diag(np.linalg.inv(J.T @ J)) * cost / (n - NPARAM))


def fit_batch(samples, offsets, padding: int, tau0: float):
    """`fit_event` + `is_valid` over a flat event buffer: (params [E, 6], cost [E], type [E] (1 valid, 7 failed))."""
    E = len(offsets) - 1
    P = np.zeros((E, NPARAM)); cost = np.zeros(E); typ = np.zeros(E, np.int32)
    for e in range(E):
        x = np.asarray(samples[offsets[e]:offsets[e + 1]], np.float64)
        p, c, conv, _ = fit_event(x, padding, tau0)
        P[e], cost[e] = p, c
        typ[e] = 1 if is_valid(p, x.size, conv, initial_guess(x, padding, tau0)[0]) else 7
    return P, cost, typ
