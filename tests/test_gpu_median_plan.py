"""The median estimate left on the device for the forward filter pass (ct_median_plan, ct_filter_forward_planned_u16).

TraceAnalyzer queues the forward pass behind the estimate's rank search and reads the estimate while the pass runs, so
  * the CtMedianPlan the rank search writes must be the MedianPlan the host arithmetic of median.estimate makes from the
    same histogram (est, window lo, standard error; the sample count of all ranks when it travels with the histogram),
    on a narrow trace, a drifting one, two levels with the sampled median off the true one, and an estimate two code
    steps off the median;
  * the pass that reads sub_code and the window's first code from it must leave the scratch, the window counts and,
    after the backward pass, the filtered trace of the by-value pass bit for bit (whole trace and streamed pieces, with
    and without the count, every scratch decimation and a one- and five-section cascade);
  * the analyzer on that route must return what it returns when the host reads the estimate first (fused_count=False).
"""
import ctypes as C

import numpy as np
import pytest
import torch

from cusumtools_b200 import _lib, filters, median, pipeline, synth
from cusumtools_b200.design import bessel_lowpass

S = synth.CHIMERA_SETTINGS
MASK = filters.chimera_bitmask(S)
PAD = 1000
N = 5_000_000
KW = dict(threshold=5.0, hysteresis=1.0, baseline_min=4700.0, baseline_max=5300.0)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def traces() -> dict:
    """The traces of the median-route tests of the analyzer (test_gpu_pipeline.py)."""
    base, _ = synth.c1_trace(n=N, n_events=600, seed=7)
    drift = (base.astype(np.int64) + 4 * (np.arange(N) * 3000 // N)).astype(np.uint16)
    srt = np.sort(base & np.uint16(MASK))
    a = int(srt[(N - 1) // 2])
    two = np.full(N, a + 160, dtype=np.uint16)          # the sampled positions hold A, the median is A + 40 steps
    two[::4] = a
    two[1::4][: N // 4 - 2] = a
    off, _ = synth.c1_trace(n=N, n_events=600, seed=11)
    off = off.copy()
    off[::4] += np.uint16(8)                            # the estimate is the median + 2 steps
    return {"narrow": base, "drift": drift, "two levels": two, "off by two": off}


@pytest.fixture(scope="module")
def trace_set():
    return traces()


def test_plan_layout_and_argument_errors_without_gpu():
    L = _lib.lib()
    assert C.sizeof(_lib.CtMedianPlan) == 56
    assert L.ct_median_plan(None, 0, 2, None, None, None) == -1
    assert L.ct_median_plan(C.c_void_p(64), 0, 17, None, C.c_void_p(64), None) == -1
    coef = filters.make_coef(bessel_lowpass(8, 2e5 / synth.FS))
    rc = L.ct_filter_forward_planned_u16(C.c_void_p(64), 10, PAD, None, MASK, 0.0, C.byref(coef), 238, 0, 0, 4, 0, 10,
                                         None, 0, 0, None, 0, None)
    assert rc == -1 and b"bad argument" in L.ct_last_error()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["narrow", "drift", "two levels", "off by two"])
def test_device_plan_is_the_host_estimate(trace_set, name):
    codes = trace_set[name]
    raw = torch.from_numpy(codes).cuda()
    hist_fn = median.device_counters(raw, MASK)[0]
    buf = median.PlanBuffer(raw.device)
    got = median.estimate_start(N, MASK, hist_fn, buf=buf).result()
    want = median.estimate(N, MASK, lambda stride: hist_fn(stride).cpu())      # the host branch, same histogram
    assert got == want
    p = _lib.CtMedianPlan.from_buffer_copy(buf.host.numpy())
    assert p.sub_code == np.float32(want.est) and p.step == want.step == 4 and p.n == 0
    # the rank search of ct_hist_rank, and the int64 histogram with the sample count of all ranks (the all_reduce form)
    h = hist_fn(N // (1 << 20))
    out = torch.empty(3, dtype=torch.int64, device="cuda")
    _lib.check(_lib.lib().ct_hist_rank(h.data_ptr(), 0, out.data_ptr(), _stream()), "ct_hist_rank")
    assert [p.bin, p.dens, p.total] == out.tolist()
    packed = torch.cat((h.to(torch.int64), torch.tensor([N + 12345], dtype=torch.int64, device="cuda")))
    dev = torch.empty(C.sizeof(_lib.CtMedianPlan), dtype=torch.uint8, device="cuda")
    _lib.check(_lib.lib().ct_median_plan(packed.data_ptr(), 1, 2, packed[-1:].data_ptr(), dev.data_ptr(), _stream()),
               "ct_median_plan")
    q = _lib.CtMedianPlan.from_buffer_copy(dev.cpu().numpy())
    assert q.n == N + 12345
    assert [getattr(q, f) for f, _ in q._fields_ if f != "n"] == [getattr(p, f) for f, _ in p._fields_ if f != "n"]


class Pass:
    """The forward pass (by value or from the device plan) and the backward pass of one trace."""

    def __init__(self, raw, design, origin):
        L = _lib.lib()
        self.raw, self.n, self.origin = raw, raw.numel(), origin
        self.coef, self.H = filters.make_coef(design), filters.warmup_samples(design)
        self.wsb = int(L.ct_filtfilt_workspace_bytes(self.n, PAD, self.H))

    def run(self, plan_dev, est, lo, pieces, count, pad_x):
        L, n = _lib.lib(), self.n
        ws = torch.zeros(self.wsb, dtype=torch.uint8, device="cuda")
        counts = torch.zeros(9, dtype=torch.int64, device="cuda")
        cb, ce = n // 7, n - n // 5                              # a time shard counts its owned samples only
        for part, a, b in pieces:
            cnt = counts.data_ptr() if count else None
            if plan_dev is None:
                rc = L.ct_filter_forward_u16(self.raw.data_ptr(), n, PAD, float(est), MASK, pad_x, C.byref(self.coef), self.H,
                                             self.origin, part, lo, 4, cb, ce, cnt, a, b, ws.data_ptr(), self.wsb, _stream())
            else:
                rc = L.ct_filter_forward_planned_u16(self.raw.data_ptr(), n, PAD, plan_dev.data_ptr(), MASK, pad_x,
                                                     C.byref(self.coef), self.H, self.origin, part, 4, cb, ce, cnt, a, b,
                                                     ws.data_ptr(), self.wsb, _stream())
            _lib.check(rc, "forward")
        y = torch.empty(n, dtype=torch.float32, device="cuda")
        alpha = filters.chimera_affine(S)[0]
        offset = float(filters.scale_codes_host(np.array([est], dtype=np.uint16), S)[0])
        _lib.check(L.ct_filter_backward(n, PAD, float(est), alpha, offset, C.byref(self.coef), self.H, self.origin, y.data_ptr(),
                                        ws.data_ptr(), self.wsb, None, None, _stream()), "ct_filter_backward")
        torch.cuda.synchronize()
        return ws[:self.wsb - 256], counts, y                   # (the last 256 bytes hold the passes' work counters)


@pytest.mark.gpu
@pytest.mark.parametrize("poles, cutoff", [(8, 1e5), (8, 2.5e5), (8, 9e5), (10, 1e5), (1, 2e5)])   # D 4 / 2 / 1, 5 and 1 sections
def test_planned_forward_pass_is_the_by_value_pass(trace_set, poles, cutoff):
    design = bessel_lowpass(poles, 2.0 * cutoff / synth.FS)
    for name in ("narrow", "drift"):
        raw = torch.from_numpy(trace_set[name]).cuda()
        buf = median.PlanBuffer(raw.device)
        plan = median.estimate_start(N, MASK, median.device_counters(raw, MASK)[0], buf=buf).result()
        for origin in (0, 777):
            ps = Pass(raw, design, origin)
            cuts = [0, N // 3, 2 * N // 3, N]
            for pieces, count, pad_x in (([(0, 0, 0)], True, 0.0), ([(2, a, b) for a, b in zip(cuts[:-1], cuts[1:])], True, 0.0),
                                         ([(0, 0, 0)], False, 1.5)):
                want = ps.run(None, plan.est, plan.lo, pieces, count, pad_x)
                got = ps.run(buf.dev, plan.est, plan.lo, pieces, count, pad_x)
                what = (name, origin, pieces[0][0], count)
                assert torch.equal(got[0], want[0]), what
                assert torch.equal(got[1], want[1]), what
                assert torch.equal(got[2].view(torch.int32), want[2].view(torch.int32)), what
                if count:
                    assert int(want[1].sum()) > 0, what


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["narrow", "drift", "two levels", "off by two"])
def test_analyzer_route_with_the_device_plan_is_the_host_read_route(trace_set, name):
    raw = torch.from_numpy(trace_set[name]).cuda()
    out = []
    for fused in (True, False):
        an = pipeline.TraceAnalyzer(N, S, 1e5, 8, baseline_block=65536, maxpoints=4000, fused_count=fused, **KW)
        r = an.run(raw)
        r = an.run(raw)                                          # a second step through the same buffers
        out.append((an.last_median_route, r.median_codes, r.pad_value, r.filtered.view(torch.int32).clone(),
                    r.events.starts.clone(), r.events.ends.clone()))
    (route, *a), (_, *b) = out
    assert route == {"narrow": "device", "drift": "host", "two levels": "host after a device miss",
                     "off by two": "device"}[name]
    assert a[0] == b[0] and a[1] == b[1]
    for x, y in zip(a[2:], b[2:]):
        assert torch.equal(x, y), name
