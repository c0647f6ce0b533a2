"""Step-response fit of short events on the GPU (ct_stepfit_select / ct_stepfit_batch, rate.csv type 1 / 7) against
its definition (oracle/stepfit_oracle.py), and its place in the pipeline: ordering with CUSUM+, the derived columns,
the streamed form, the default (off) path and the two-GPU sharded run."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from cusumtools_b200 import pipeline, stepfit, synth, writer
from oracle import stepfit_oracle as so

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FS = synth.FS
PAD = synth.SHORT_PAD
TAU0 = stepfit.zero_phase_rise_tau(FS, 1e5, 8)
S = synth.CHIMERA_SETTINGS
KW = dict(threshold=5.0, hysteresis=1.0, baseline_block=1 << 16, baseline_min=4700.0, baseline_max=5300.0,
          cusum_delta=400.0, cusum_h=10.0)


@pytest.fixture(scope="module")
def short_events():
    x, off, lens, depth = synth.short_events_device(2000, "cuda:0", seed=11)
    t = stepfit.stepfit_flat(x, off, padding=PAD, tau0=TAU0)
    torch.cuda.synchronize()
    xs, of = x.cpu().numpy(), off.cpu().numpy()
    P, cost, typ = so.fit_batch(xs, of, PAD, TAU0)
    return dict(x=xs, off=of, lens=lens.cpu().numpy(), depth=depth.cpu().numpy(), t=t, P=P, cost=cost, typ=typ)


def test_kernel_matches_oracle(short_events):
    d = short_events
    t = d["t"]
    gt, gp, gc = t.status.cpu().numpy(), t.params.cpu().numpy(), t.cost.cpu().numpy()
    assert set(np.unique(gt)) <= {1, 7}
    agree = gt == d["typ"]
    # the two solvers take different paths; on about 2 % of the events (mostly the shortest, where a and tau trade off)
    # one of them ends at max_iters or at another local minimum and the type differs
    assert agree.mean() >= 0.97, f"type 1/7 differs on {np.count_nonzero(~agree)} of {agree.size}: {np.nonzero(~agree)[0][:10]}"
    both = np.nonzero((gt == 1) & (d["typ"] == 1))[0]
    assert both.size > 0.9 * gt.size
    cost_ok = gc[both] <= d["cost"][both] * (1 + 1e-5)
    dev = np.array([np.max(np.abs(gp[e] - d["P"][e]) / so.standard_errors(d["x"][d["off"][e]:d["off"][e + 1]].astype(np.float64),
                                                                           d["P"][e])) for e in both])
    # where both fit, the median parameter difference is ~1e-3 se; 7-8 % of the events end in a different local
    # minimum of the kinked cost surface (u at a sample boundary, a against tau on the shortest events)
    assert cost_ok.mean() >= 0.95, np.percentile(gc[both] / d["cost"][both], [50, 95, 99])
    assert np.median(dev) <= 0.01 and np.mean(dev <= 0.05) >= 0.90, np.percentile(dev, [50, 90, 95, 99])
    # the level rows of every valid fit
    lv = t.levels
    nl, ed, mu, sd = (v.cpu().numpy() for v in (lv.n_levels, lv.edges, lv.mean, lv.std))
    for e in both[:50]:
        x = d["x"][d["off"][e]:d["off"][e + 1]].astype(np.float64)
        edges, mean, std = so.level_rows(x, gp[e])
        assert nl[e] == 3 and np.array_equal(ed[e, :4], edges)
        assert np.allclose(mu[e, :3], mean, rtol=1e-12) and np.allclose(sd[e, :3], std, rtol=1e-4, atol=1e-3)
    assert np.all(nl[gt == 7] == 0)


def test_noise_free_windows_are_recovered():
    rng = np.random.default_rng(3)
    rows, wins = [], []
    for k in range(300):
        L = int(rng.integers(60, 600))
        n = L + 2 * PAD
        sgn = 1.0 if k % 2 == 0 else -1.0
        p = np.array([sgn * 5000.0 + rng.uniform(-50, 50), sgn * rng.uniform(300, 2000), PAD + rng.uniform(-3, 3),
                      n - PAD + rng.uniform(-3, 3), rng.uniform(8, 30), rng.uniform(8, 30)])
        rows.append(p)
        wins.append(so.model(p, n).astype(np.float32))
    off = np.concatenate(([0], np.cumsum([w.size for w in wins]))).astype(np.int64)
    x = torch.from_numpy(np.concatenate(wins)).cuda()
    t = stepfit.stepfit_flat(x, torch.from_numpy(off).cuda(), padding=PAD, tau0=TAU0)
    P = np.array(rows)
    assert np.all(t.status.cpu().numpy() == 1)
    rel = np.abs(t.params.cpu().numpy() - P) / np.abs(P)
    assert rel.max() <= 1e-4, rel.max(axis=0)


def test_select_kernel():
    cap = 64
    w0 = torch.arange(cap, dtype=torch.int64, device="cuda") * 10_000
    lengths = torch.tensor([5, 99, 100, 101, 400] * 12 + [1, 2, 3, 50], dtype=torch.int64, device="cuda")
    w1 = w0 + lengths + 2 * PAD
    types = torch.tensor([0, 0, 0, 0, 2, 3, 4, 0] * 8, dtype=torch.int32, device="cuda")
    count = torch.tensor([40], dtype=torch.int64, device="cuda")
    out = types.clone()
    stepfit.select_short(w0, w1, out, padding=PAD, stepfit_samples=100, n_events_dev=count)
    got, t0, ln = out.cpu().numpy(), types.cpu().numpy(), lengths.cpu().numpy()
    want = t0.copy()
    want[:40][(t0[:40] == 0) & (ln[:40] < 100)] = 1
    assert np.array_equal(got, want)                   # rows at or beyond the count are untouched
    assert np.array_equal(got[t0 > 1], t0[t0 > 1])     # types 2/3/4 stay


def test_event_columns_of_type1_rows_match_host(short_events):
    d = short_events
    x = torch.from_numpy(d["x"]).cuda()
    off = torch.from_numpy(d["off"]).cuda()
    w0, w1 = off[:-1].contiguous(), off[1:].contiguous()
    t = stepfit.step_fit(x, w0, w1, padding=PAD, tau0=TAU0)
    lo, hi = writer.event_extrema(x, w0, w1)
    cols, tout = writer.event_columns(t.levels, t.status, lo, hi)
    lv = t.levels
    hc, ht = writer.event_columns_host(t.status.cpu().numpy(), lv.n_levels.cpu().numpy(), lv.edges.cpu().numpy(),
                                       lv.mean.cpu().numpy(), lv.std.cpu().numpy(), lv.overflow.cpu().numpy(),
                                       lo.cpu().numpy(), hi.cpu().numpy())
    assert np.array_equal(tout.cpu().numpy(), ht)
    assert np.allclose(cols.cpu().numpy(), hc, rtol=1e-12, atol=1e-9)
    ok = ht == 1
    p = t.params.cpu().numpy()[ok]
    assert np.allclose(hc[ok, 5], np.abs(p[:, 1]), rtol=1e-12)          # max_blockage = |a|
    assert np.allclose(hc[ok, 7], np.abs(p[:, 1]), rtol=1e-12)          # min_blockage = |a|


def _pulse_trace(L: int, seed: int, n: int = 4_194_304, depth: float = -1000.0):
    return synth.device_trace(n, "cuda:0", seed=seed, levels=((depth, L),))


def _run(codes, **kw):
    an = pipeline.TraceAnalyzer(codes.numel(), S, 1e5, 8, device="cuda:0", **KW, **kw)
    r = an.run(codes)
    tab = writer.event_table_from_result(an, r, samplerate=FS)
    return an, r, tab


@pytest.mark.parametrize("L", [30, 100, 200, 400])
def test_pipeline_short_pulses_become_type1(L):
    codes = _pulse_trace(L, seed=100 + L)
    _, r_off, tab_off = _run(codes)
    an, r_on, tab_on = _run(codes, stepfit_samples=500)
    assert np.array_equal(tab_on.rate["start_time_s"], tab_off.rate["start_time_s"])
    t_off, t_on = tab_off.rate["type"], tab_on.rate["type"]
    short = np.isin(t_off, (0, 5))
    assert short.sum() > 900
    assert np.all(np.isin(t_on[short], (1, 7))) and np.mean(t_on[short] == 1) > (0.95 if L >= 100 else 0.85)
    assert np.array_equal(t_on[~short], t_off[~short])
    # ordering: the level rows of the fitted events survived the CUSUM+ launch that ran before the fit
    nl = r_on.levels.n_levels.cpu().numpy()
    typ = r_on.types.cpu().numpy()
    p = r_on.stepfit.params.cpu().numpy()
    mu = r_on.levels.mean.cpu().numpy()
    assert np.all(nl[typ == 1] == 3) and np.allclose(mu[typ == 1, 1], p[typ == 1, 0] - p[typ == 1, 1])
    ev = tab_on.events
    fitted = ev["type"] == 1
    assert np.all(ev["rc_const1_us"][fitted] > 0) and np.all(ev["rc_const1_us"][~fitted] == 0)
    assert np.allclose(ev["rc_const1_us"][fitted], p[typ == 1, 4] * 1e6 / FS)
    err_on = np.abs(ev["max_blockage_pA"][fitted] - 1000.0) / 1000.0
    if L >= 100:
        assert np.median(err_on) <= 0.02, np.median(err_on)
        ok_off = tab_off.events["type"] == 0
        err_off = np.abs(tab_off.events["max_blockage_pA"][ok_off] - 1000.0) / 1000.0
        assert np.median(err_on) < np.median(err_off) if ok_off.any() else True
    else:
        # a and tau trade off against each other this short: type and oracle parity only
        y = r_on.detect_trace.cpu().numpy()
        w0, w1 = r_on.win_start.cpu().numpy(), r_on.win_end.cpu().numpy()
        sel = np.nonzero(np.isin(typ, (1, 7)))[0][:200]
        same = []
        for i in sel:
            x = y[w0[i]:w1[i]].astype(np.float64)
            q, _, conv, _ = so.fit_event(x, PAD, an.tau0)
            same.append((typ[i] == 1) == so.is_valid(q, x.size, conv, so.initial_guess(x, PAD, an.tau0)[0]))
        assert np.mean(same) >= 0.85, np.mean(same)         # 0.88 measured on this trace


def test_streamed_form_gives_the_same_stepfit_columns():
    codes = _pulse_trace(150, seed=7)
    an, r, _ = _run(codes, stepfit_samples=500)
    res = an.tables_to_host(r)
    res = {k: v.copy() for k, v in res.items()}
    n = codes.numel()
    san = pipeline.StreamingAnalyzer(n, S, 1e5, 8, shards=3, first_blocks=2, device="cuda:0", stepfit_samples=500, **KW)
    rs = san.run_from_host(codes.cpu().pin_memory())
    t = rs.tables
    assert np.array_equal(t["starts"], res["starts"]) and np.array_equal(t["types"], res["types"])
    both = res["types"] == 1
    assert both.sum() > 900
    dp = np.abs(t["stepfit_params"][both] - res["stepfit_params"][both])
    assert np.percentile(dp[:, 1], 99) < 0.5 and np.percentile(dp[:, 2:], 99) < 0.05, dp.max(axis=0)
    assert np.all(t["stepfit_iters"][~both] == 0) and np.all(t["stepfit_params"][~both] == 0)


def test_default_is_unchanged():
    codes = _pulse_trace(150, seed=9)
    a0 = pipeline.TraceAnalyzer(codes.numel(), S, 1e5, 8, device="cuda:0", **KW)
    a1 = pipeline.TraceAnalyzer(codes.numel(), S, 1e5, 8, device="cuda:0", stepfit_samples=0, **KW)
    r0, r1 = a0.run(codes), a1.run(codes)
    h0, h1 = a0.tables_to_host(r0), a1.tables_to_host(r1)
    assert r1.stepfit is None and sorted(h0) == sorted(h1)
    nl = h0["n_levels"]
    written = np.arange(h0["mean"].shape[1])[None, :] < nl[:, None]          # level entries the kernels write
    for k in h0:
        if k in ("mean", "std"):
            assert np.array_equal(h0[k][written], h1[k][written]), k
        else:
            assert np.array_equal(h0[k], h1[k]), k
    assert torch.equal(r0.filtered, r1.filtered)


def test_window_limit_is_checked():
    with pytest.raises(ValueError, match="window"):
        pipeline.TraceAnalyzer(1 << 20, S, 1e5, 8, device="cuda:0", stepfit_samples=stepfit.MAX_WINDOW, **KW)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_sharded_stepfit_equals_unsharded_on_two_gpus():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29733", os.path.join(ROOT, "scripts", "check_sharded.py"), "--stepfit-samples", "500"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "OK" in out.stdout and "stepfit" in out.stdout
