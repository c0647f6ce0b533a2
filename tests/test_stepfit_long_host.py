"""Long windows (8 k - 131 k samples, the range of the long step-fit kernel) through the float64 twin of the fit's LM
loop (oracle/stepfit_twin.py), without a GPU: noise-free parameters are recovered and every valid fit of a filtered
shallow pulse is a local minimum scipy's float64 LM cannot improve.  Also: the template cycle of synth.device_trace
leaves the single-template traces as they were."""
import numpy as np
import pytest
import torch

from cusumtools_b200 import synth
from oracle import stepfit_oracle as so
from oracle import stepfit_twin as tw

FS = 4166666.0
PAD = 100
TAU0 = 38 / np.log(9.0)          # stepfit.zero_phase_rise_tau(FS, 1e5, 8)


@pytest.mark.parametrize("n", [8193, 20_000, 100_200, 131_072])
def test_noise_free_long_windows_are_recovered(n):
    rng = np.random.default_rng(n)
    for k in range(4):
        sgn = 1.0 if k % 2 else -1.0
        p = np.array([sgn * 5000 + rng.uniform(-30, 30), sgn * rng.uniform(120, 2000), PAD + rng.uniform(-2, 2),
                      n - PAD + rng.uniform(-2, 2), rng.uniform(8, 30), rng.uniform(8, 30)])
        x = so.model(p, n).astype(np.float32)
        f = tw.fit(x, PAD, TAU0)
        assert f.type == 1 and f.converged, (n, k, f.iters, f.params, p)
        # i0 and u within 1e-6 relative as for short windows (test_stepfit_twin_host); a within 3e-6 and the rise
        # times within 1e-5 (measured 1.1e-6 and 4.0e-6: steps down to 120 pA, where the float32 rounding of the
        # +-5000 pA samples is a larger share of the step, and windows up to 131 072 samples, whose stop floor
        # n (2^-24 max|x - x0|)^2 grows with n)
        rel = np.abs(f.params - p) / np.abs(p)
        assert rel[0] <= 1e-6 and rel[2] <= 1e-6 and rel[3] <= 1e-6, (n, k, rel)
        assert rel[1] <= 3e-6 and np.all(rel[4:] <= 1e-5), (n, k, rel)


def shallow_pulses(lengths, depth_lo, depth_hi, seed, noise=150.0, guard=400):
    """Filtered rectangular pulses (scipy bessel + filtfilt, 100 kHz / 8 poles) of the given lengths with PAD baseline
    samples either side, depth uniform in [depth_lo, depth_hi] pA toward zero from +-5000 pA."""
    from scipy import signal
    rng = np.random.default_rng(seed)
    b, a = signal.bessel(8, 2.0 * 1e5 / FS)
    out = []
    for k, L in enumerate(lengths):
        sgn = 1.0 if k % 2 == 0 else -1.0
        x = np.full(int(L) + 2 * PAD + 2 * guard, sgn * 5000.0)
        x[guard + PAD:guard + PAD + int(L)] -= sgn * rng.uniform(depth_lo, depth_hi)
        x += noise * rng.standard_normal(x.size)
        out.append(signal.filtfilt(b, a, x)[guard:guard + int(L) + 2 * PAD].astype(np.float32))
    return out


def test_valid_fits_of_shallow_long_pulses_are_local_minima():
    rng = np.random.default_rng(3)
    lengths = np.exp(rng.uniform(np.log(8000), np.log(100_000), 8)).astype(np.int64)
    n_valid, worst = 0, (0.0, 0.0)
    for x in shallow_pulses(lengths, 120.0, 200.0, seed=4):
        f = tw.fit(x, PAD, TAU0)
        if f.type != 1:
            continue
        n_valid += 1
        e, m, s = so.level_rows(x, f.params)
        assert np.array_equal(f.edges, e) and np.allclose(f.mean, m, rtol=1e-12) and np.allclose(f.std, s, rtol=1e-9)
        dc, move = tw.local_minimum_gap(x, f.params)
        worst = max(worst[0], dc), max(worst[1], move)
    assert n_valid >= 0.85 * len(lengths)
    assert worst[0] <= 1e-6 and worst[1] <= 0.02, worst


def _parent_device_trace(n, seed, levels):
    """device_trace's signal model for one template, restated (CPU): the noise stream of the seed, every event k at
    1500 + k period + jitter_k with the template's levels, quantised as synth.quantise's torch form."""
    g = torch.Generator(device="cpu")
    g.manual_seed(seed)
    alpha, beta = synth._affine(synth.CHIMERA_SETTINGS)
    step = 1 << (16 - 14)
    period = int(round(synth.FS / 1000.0))
    cur = torch.randn(n, generator=g, dtype=torch.float32) * synth.NOISE_PA + synth.BASELINE_PA
    gidx = torch.arange(n, dtype=torch.int64)
    k = torch.div(gidx - 1500 + 500, period, rounding_mode="floor")
    for kk in (k, k - 1):
        h = (kk * 2654435761) % 4294967296
        st = 1500 + kk * period + (h % 1001) - 500
        rel = gidx - st
        o = 0
        for depth, length in levels:
            cur += depth * ((rel >= o) & (rel < o + length) & (kk >= 0))
            o += length
    code = torch.round((cur - beta) / alpha / step) * step
    return code.clamp_(0, 65536 - step).to(torch.int32).to(torch.uint16)


def test_template_cycle_keeps_single_template_traces():
    n = 200_000
    pulse = ((-1000.0, 100),)
    default = synth.device_trace(n, "cpu", seed=11)
    assert torch.equal(default, _parent_device_trace(n, 11, synth.EVENT_LEVELS))
    assert torch.equal(synth.device_trace(n, "cpu", seed=11, levels=pulse), _parent_device_trace(n, 11, pulse))
    assert torch.equal(synth.device_trace(n, "cpu", seed=11, levels=[synth.EVENT_LEVELS]), default)
    # two templates: event k takes template k mod 2, the noise stream is the seed's either way
    mixed = synth.device_trace(n, "cpu", seed=11, levels=[synth.EVENT_LEVELS, pulse]).numpy()
    only_pulse = synth.device_trace(n, "cpu", seed=11, levels=pulse).numpy()
    period = int(round(synth.FS / 1000.0))
    for k in range(int(n // period) - 1):
        lo, hi = 1000 + k * period, 1000 + (k + 1) * period     # event k lies inside [lo, hi)
        want = default if k % 2 == 0 else only_pulse
        assert np.array_equal(mixed[lo:hi], np.asarray(want)[lo:hi]), k
