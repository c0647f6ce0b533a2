"""The float64 twin of the step-fit kernel's LM loop (oracle/stepfit_twin.py) without a GPU: it recovers noise-free
parameters, stops where the kernel stops, and every valid fit it makes on filtered pulses is a local minimum that
scipy's float64 LM cannot improve."""
import numpy as np
import pytest

from oracle import stepfit_oracle as so
from oracle import stepfit_twin as tw

FS = 4166666.0
PAD = 100
TAU0 = 38 / np.log(9.0)          # stepfit.zero_phase_rise_tau(FS, 1e5, 8)


def filtered_pulses(n_events: int, min_len: int, max_len: int, seed: int):
    """Filtered rectangular pulses of log-uniform length in [min_len, max_len] samples, each with PAD baseline samples
    either side (stepfit_twin.filtered_pulse_windows)."""
    rng = np.random.default_rng(seed)
    L = np.exp(rng.uniform(np.log(min_len), np.log(max_len), n_events)).astype(np.int64)
    return tw.filtered_pulse_windows(L + 2 * PAD, PAD, seed)


def noise_free(k: int, rng, n_lo=80, n_hi=500):
    L = int(rng.integers(n_lo, n_hi))
    n = L + 2 * PAD
    sgn = 1.0 if k % 2 else -1.0
    p = np.array([sgn * 5000 + rng.uniform(-30, 30), sgn * rng.uniform(300, 2000), PAD + rng.uniform(-2, 2),
                  n - PAD + rng.uniform(-2, 2), rng.uniform(8, 30), rng.uniform(8, 30)])
    return p, so.model(p, n).astype(np.float32)


def test_noise_free_windows_are_recovered():
    rng = np.random.default_rng(5)
    for k in range(20):
        p, x = noise_free(k, rng)
        f = tw.fit(x, PAD, TAU0)
        assert f.type == 1 and f.converged, (k, f.iters, f.params, p)
        # the stop floor n (2^-24 max|x - x0|)^2 ends the fit within float32 resolution of the cost, which leaves the
        # rise times (the flattest directions) up to 1.7e-6 relative from the truth on these windows (i0, a, u: 7e-7)
        rel = np.abs(f.params - p) / np.abs(p)
        assert np.all(rel[:4] <= 1e-6) and np.all(rel[4:] <= 5e-6), rel


def test_one_trial_returns_the_initial_guess_as_type7():
    rng = np.random.default_rng(6)
    p, x = noise_free(0, rng)
    f = tw.fit(x, PAD, TAU0, max_iters=1)
    assert f.iters == 1 and f.type == 7 and not f.converged and f.steps == []
    assert np.array_equal(f.params, f.initial)
    xr, x0 = tw.window(x)
    assert np.array_equal(f.initial, tw.initial_point(xr, PAD, TAU0) + np.array([x0, 0, 0, 0, 0, 0]))
    assert f.initial[4] == float(np.float32(TAU0)) and np.isclose(f.cost, tw.cost_at(x, f.params), rtol=1e-12)


def test_initial_guess_is_the_definitions():
    x = filtered_pulses(1, 100, 101, seed=1)[0]
    f = tw.fit(x, PAD, TAU0, max_iters=1)
    want = so.initial_guess(x, PAD, TAU0)
    assert np.allclose(f.initial[:4], want[:4], rtol=1e-12, atol=1e-9) and np.allclose(f.initial[4:], TAU0, rtol=1e-7)


def test_flat_window_never_has_a_step():
    for level in (5000.0, -5000.0, 0.0):
        f = tw.fit(np.full(300, level, np.float32), PAD, TAU0)
        # a = 0: the u and tau columns of J vanish, no matrix is positive definite, mu grows x10 per trial until it
        # reaches 1e30 (1e-3 x 10^33 rounds below 1e30: 34 unevaluated trials)
        assert f.type == 7 and not f.converged and all(s.kind == "no_pd" for s in f.steps)
        assert f.iters == 35 and np.all(np.isfinite(f.params)) and f.cost == 0.0


def test_trial_counter_counts_unevaluated_trials():
    rng = np.random.default_rng(8)
    for k in range(10):
        _, x = noise_free(k, rng)
        f = tw.fit(x, PAD, TAU0)
        evaluated = sum(s.kind in ("accept", "reject") for s in f.steps)
        unevaluated = sum(s.kind in ("no_pd", "domain") for s in f.steps)
        assert f.iters == 1 + evaluated + unevaluated


@pytest.mark.parametrize("lengths", [(20, 400), (800, 7700)])
def test_valid_fits_of_filtered_pulses_are_local_minima(lengths):
    xs = filtered_pulses(40 if lengths[0] < 100 else 12, *lengths, seed=lengths[0])
    n_valid, worst = 0, (0.0, 0.0)
    for x in xs:
        f = tw.fit(x, PAD, TAU0)
        assert np.isclose(f.cost, tw.cost_at(x, f.params), rtol=1e-9)
        if f.type != 1:
            continue
        n_valid += 1
        assert np.array_equal(f.edges, [0, np.ceil(f.params[2]), np.ceil(f.params[3]), x.size])
        e, m, s = so.level_rows(x, f.params)
        assert np.array_equal(f.edges, e) and np.allclose(f.mean, m, rtol=1e-12) and np.allclose(f.std, s, rtol=1e-9)
        dc, move = tw.local_minimum_gap(x, f.params)
        worst = max(worst[0], dc), max(worst[1], move)
    assert n_valid >= 0.85 * len(xs)
    assert worst[0] <= 1e-6 and worst[1] <= 0.02, worst
