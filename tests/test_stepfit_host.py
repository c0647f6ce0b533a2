"""The step-response fit of short events without a GPU: the oracle's model, initial guess and validity rule
(oracle/stepfit_oracle.py), the type-1 rows of the derived columns (writer.event_columns_host), and type-1 events
through events.csv / rate.csv / summary.txt / the 4-column event file and back through the consumers' parsing
statements (readevents.py:73-79,1318-1337; plot-trace.py:181-203,354-357), as test_writer.py does for type 0."""
import math
import os
import re

import numpy as np
import pandas as pd

from cusumtools_b200 import stepfit, writer
from oracle import stepfit_oracle as so

FS = 4166666.0
PAD, BLOCK = 100, 65536
TAU0 = 17.29


def test_tau0_is_the_zero_phase_rise_time():
    assert abs(stepfit.zero_phase_rise_tau(FS, 1e5, 8) - 38 / math.log(9)) < 1e-12


def test_oracle_recovers_noise_free_parameters():
    rng = np.random.default_rng(1)
    for k in range(20):
        L = int(rng.integers(80, 500))
        n = L + 2 * PAD
        sgn = 1.0 if k % 2 else -1.0
        p = np.array([sgn * 5000 + rng.uniform(-30, 30), sgn * rng.uniform(300, 2000), PAD + rng.uniform(-2, 2),
                      n - PAD + rng.uniform(-2, 2), rng.uniform(8, 30), rng.uniform(8, 30)])
        q, cost, conv, _ = so.fit_event(so.model(p, n), PAD, TAU0)
        assert conv and np.all(np.abs(q - p) <= 1e-6 * np.abs(p)), (q, p)
        assert so.is_valid(q, n, conv, so.initial_guess(so.model(p, n), PAD, TAU0)[0])


def test_jacobian_is_the_derivative_of_the_model():
    p = np.array([5000.0, 800.0, 100.4, 300.6, 15.0, 20.0])
    J = so.jacobian(p, 500)
    for k in range(6):
        h = 1e-6 * max(1.0, abs(p[k]))
        dp = np.zeros(6); dp[k] = h
        num = (so.model(p + dp, 500) - so.model(p - dp, 500)) / (2 * h)
        far = np.abs(np.arange(500) - p[2]) > 1 if k == 2 else (np.abs(np.arange(500) - p[3]) > 1 if k == 3 else slice(None))
        assert np.allclose(J[far, k], num[far], rtol=1e-5, atol=1e-6 * np.abs(num).max())


def test_initial_guess_and_validity_rule():
    x = np.full(400, 5000.0)
    x[PAD:400 - PAD] = 4000.0
    g = so.initial_guess(x, PAD, TAU0)
    assert np.allclose(g, [5000.0, 1000.0, PAD, 400 - PAD, TAU0, TAU0])
    ok = np.array([5000.0, 1000.0, 100.5, 300.5, 17.0, 17.0])
    assert so.is_valid(ok, 400, True, 5000.0)
    assert not so.is_valid(ok, 400, False, 5000.0)                       # not converged
    wrong_sign = ok.copy(); wrong_sign[1] = -1000.0
    assert not so.is_valid(wrong_sign, 400, True, 5000.0)                 # current moves away from zero
    neg = ok.copy(); neg[0], neg[1] = -5000.0, -1000.0
    assert so.is_valid(neg, 400, True, -5000.0)                           # negative baseline: a < 0 is the blockage
    assert not so.is_valid(neg, 400, True, 5000.0)
    crossed = ok.copy(); crossed[2], crossed[3] = 300.5, 100.5
    assert not so.is_valid(crossed, 400, True, 5000.0)                    # u1 >= u2
    same = ok.copy(); same[2], same[3] = 100.2, 100.7
    assert not so.is_valid(same, 400, True, 5000.0)                       # no sample at the blocked level
    for tau in (0.01, 401.0):
        bad = ok.copy(); bad[5] = tau
        assert not so.is_valid(bad, 400, True, 5000.0)                    # tau outside [0.05, n]
    late = ok.copy(); late[3] = 399.5
    assert not so.is_valid(late, 400, True, 5000.0)                       # u2 leaves no sample after the event
    assert not so.in_domain(crossed) and not so.in_domain(np.r_[ok[:4], 0.0, 17.0])


def make_type1_tables(n_events=30, seed=2):
    """A trace of short pulses fitted by the oracle, laid out as the analyzer's tables (types 1, 7, 2)."""
    rng = np.random.default_rng(seed)
    period = 3000
    n = period * (n_events + 2)
    y = np.full(n, 5000.0)
    starts, ends, truth = [], [], []
    for k in range(n_events):
        s = 1500 + period * k
        L = int(rng.integers(60, 300))
        p = np.array([0.0, 900.0 + 20 * k, PAD + 0.3, L + PAD + 0.6, 16.0, 18.0])
        w = so.model(p, L + 2 * PAD)
        y[s - PAD:s + L + PAD] += w
        starts.append(s); ends.append(s + L); truth.append(p)
    y += 30.0 * rng.standard_normal(n)
    starts, ends = np.array(starts), np.array(ends)
    E = n_events
    types = np.ones(E, np.int32)
    types[3] = 2                                                          # a too-short glitch
    ML = 16
    nl = np.zeros(E, np.int32); ed = np.full((E, ML + 1), -1, np.int32); mu = np.zeros((E, ML)); sd = np.zeros((E, ML))
    params = np.zeros((E, 6))
    for i in range(E):
        if types[i] != 1:
            continue
        x = y[starts[i] - PAD:ends[i] + PAD]
        p, _, conv, _ = so.fit_event(x, PAD, TAU0)
        if not so.is_valid(p, x.size, conv, so.initial_guess(x, PAD, TAU0)[0]):
            types[i] = 7
            continue
        params[i] = p
        e, m, s_ = so.level_rows(x, p)
        nl[i] = 3; ed[i, :4] = e; mu[i, :3] = m; sd[i, :3] = s_
    w0, w1 = starts - PAD, ends + PAD
    xmin = np.array([y[a:b].min() for a, b in zip(w0, w1)], np.float32)
    xmax = np.array([y[a:b].max() for a, b in zip(w0, w1)], np.float32)
    mean = np.full(n // BLOCK + 1, 5000.0); std = np.full(n // BLOCK + 1, 30.0)
    return y, dict(s=starts, e=ends, w0=w0, w1=w1, typ=types, nl=nl, ed=ed, mu=mu, sd=sd, params=params, xmin=xmin,
                   xmax=xmax, mean=mean, std=std)


def test_event_columns_host_type1_rows():
    y, d = make_type1_tables()
    ov = np.zeros(len(d["s"]), np.uint8)
    cols, typ = writer.event_columns_host(d["typ"], d["nl"], d["ed"], d["mu"], d["sd"], ov, d["xmin"], d["xmax"])
    fit = np.nonzero(typ == 1)[0]
    assert fit.size >= 25 and np.array_equal(typ, d["typ"])
    for i in fit:
        p = d["params"][i]
        x = y[d["w0"][i]:d["w1"][i]]
        r = x - so.model(p, x.size)
        assert abs(cols[i, 5] - abs(p[1])) < 1e-9 and abs(cols[i, 7] - abs(p[1])) < 1e-9 and abs(cols[i, 4] - abs(p[1])) < 1e-9
        assert abs(cols[i, 9] - np.sqrt(np.mean(r * r))) < 1e-9 * np.sqrt(np.mean(r * r)) + 1e-12     # residual = rms(x - f)
        dur = math.ceil(p[3]) - math.ceil(p[2])
        assert cols[i, 3] == dur
        assert abs(cols[i, 4] * cols[i, 3] / FS - abs(p[1]) * dur / FS) < 1e-15                        # area_pC
    assert np.all(cols[typ > 1] == 0)


def test_type1_events_round_trip_through_the_consumers(tmp_path):
    y, d = make_type1_tables()
    tab = writer.build_event_table(starts=d["s"], ends=d["e"], types=d["typ"], n_levels=d["nl"], edges=d["ed"],
                                   level_mean=d["mu"], level_std=d["sd"], overflow=np.zeros(len(d["s"]), np.uint8),
                                   xmin=d["xmin"], xmax=d["xmax"], samplerate=FS, threshold=5.0, baseline_mean=d["mean"],
                                   baseline_std=d["std"], baseline_block=BLOCK, padding=PAD, stepfit_params=d["params"])
    ev = tab.events
    fit = d["typ"] == 1
    assert np.array_equal(ev["type"], d["typ"][fit]) and np.all(ev["n_levels"] == 2)
    assert np.allclose(ev["rc_const1_us"], d["params"][fit, 4] * 1e6 / FS, rtol=1e-15)
    assert np.allclose(ev["rc_const2_us"], d["params"][fit, 5] * 1e6 / FS, rtol=1e-15)
    assert np.allclose(ev["max_blockage_pA"], np.abs(d["params"][fit, 1]))
    i = int(np.nonzero(fit)[0][0])
    eid = int(tab.rate["id"][i])
    samples = {eid: (int(d["w0"][i]), y[d["w0"][i]:d["w1"][i]], d["ed"][i, :4].astype(np.int64), d["mu"][i, :3], d["params"][i])}
    out = str(tmp_path / "analysis")
    writer.write_analysis_dir(out, tab, baseline_mean=d["mean"], baseline_std=d["std"], baseline_block=BLOCK,
                              samplerate=FS, threshold=5.0, hysteresis=1.0, cutoff=100000.0, poles=8,
                              extra_summary={"cusum_delta": 400.0, "cusum_h": 10.0}, event_samples=samples,
                              stepfit_samples=500)
    eventsdb = pd.read_csv(os.path.join(out, "events.csv"), encoding="utf-8")
    ratedb = pd.read_csv(os.path.join(out, "rate.csv"), encoding="utf-8")
    assert list(eventsdb.columns) == writer.EVENT_COLUMNS and len(eventsdb) == int(fit.sum())
    assert np.allclose(eventsdb["rc_const1_us"].values, d["params"][fit, 4] * 1e6 / FS, rtol=1e-15)
    assert set(ratedb["type"]) == {1, 2} | ({7} if (d["typ"] == 7).any() else set())
    # readevents.py:1318-1337: type 1 -> time, current, cusum, stepfit, read with an implicit header
    event_file = pd.read_csv(os.path.join(out, "events", "event_%08d.csv" % eid), encoding="utf-8")
    event_file.columns = ["time", "current", "cusum", "stepfit"]
    x = y[d["w0"][i]:d["w1"][i]]
    assert len(event_file) == x.size                                                      # no sample lost
    assert np.allclose(event_file["current"].values, x, rtol=1e-15)
    assert np.allclose(event_file["stepfit"].values, so.model(d["params"][i], x.size), rtol=1e-12)
    e = d["ed"][i]
    assert np.all(event_file["cusum"].values[e[1]:e[2]] == d["mu"][i, 1])
    # plot-trace.py:354-357: types 0 and 1 are good
    good = ratedb[ratedb.type.isin([0, 1])]
    bad = ratedb[ratedb.type > 1]
    assert len(good) == len(eventsdb) and len(good) + len(bad) == len(ratedb)
    # summary.txt, both consumers' substring parsing (plot-trace.py:190-203, readevents.py:73-79)
    lines = open(os.path.join(out, "summary.txt")).read().splitlines()
    assert "stepfit_samples=500" in lines
    threshold = hysteresis = cutoff = poles = it = ih = None
    for line in lines:
        line += "\n"
        if "threshold" in line and "intra" not in line:
            threshold = float(re.split("=|\n", line)[1])
        if "hysteresis" in line and "intra" not in line:
            hysteresis = float(re.split("=|\n", line)[1])
        if "cutoff" in line:
            cutoff = int(re.split("=|\n", line)[1])
        if "poles" in line:
            poles = int(re.split("=|\n", line)[1])
        if "intra_threshold" in line:
            it = float(re.split("=|\n", line)[1])
        if "intra_hysteresis" in line:
            ih = float(re.split("=|\n", line)[1])
    assert (threshold, hysteresis, cutoff, poles, it, ih) == (5.0, 1.0, 100000, 8, 0.0, 0.0)


def test_type0_rows_keep_zero_rc_columns():
    y, d = make_type1_tables(n_events=8)
    typ = d["typ"].copy()
    typ[typ == 1] = 0
    tab = writer.build_event_table(starts=d["s"], ends=d["e"], types=typ, n_levels=d["nl"], edges=d["ed"],
                                   level_mean=d["mu"], level_std=d["sd"], overflow=np.zeros(len(d["s"]), np.uint8),
                                   xmin=d["xmin"], xmax=d["xmax"], samplerate=FS, threshold=5.0, baseline_mean=d["mean"],
                                   baseline_std=d["std"], baseline_block=BLOCK, padding=PAD, stepfit_params=d["params"])
    assert np.all(tab.events["type"] == 0) and np.all(tab.events["rc_const1_us"] == 0) and np.all(tab.events["rc_const2_us"] == 0)
