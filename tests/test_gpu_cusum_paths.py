"""CUSUM+ (csrc/ct_cusum.cu) on every path of its two kernels, bit for bit against the C twin.

The cases come from tests/cusum_cases.py, whose witnesses (checked on the host by tests/test_cusum_cases_host.py) show
that each reaches the path it is named for.  Here every case runs through the C ABI with a workspace of the test's
own, so that the pending list tells which kernel took each window: the thread-per-event kernel (lanes) or the
warp-per-event kernel (warps).  Each case runs with the trace 16-byte aligned (the lanes take the batch) and one float
off (the warps take everything).  n_levels, edges and overflow are compared for every row, mean and std up to
n_levels; outputs start from sentinel values, so a row the kernels should write and do not is seen too."""
import numpy as np
import pytest
import torch

import cusum_cases as cc
from cusumtools_b200 import _lib

pytestmark = pytest.mark.gpu

WS_HEAD = 544                   # kWsHead, see the layout comment above ct_cusum_workspace_bytes in csrc/ct_cusum.cu
SENT_NL, SENT_OVF, SENT_F64 = -7, 0xA5, -1234.5
LANES_AND_WARPS = (0, 1)        # trace offsets in floats


def pending_rows(ws: torch.Tensor) -> np.ndarray:
    """Rows the lanes left to the warps, read from the workspace (layout: the comment above ct_cusum_workspace_bytes):
    the pending count is the uint64 counter[1] at bytes 8-16, the pending list is int32 from byte WS_HEAD."""
    w = ws.cpu().numpy()
    n = int(w[:6].view(np.int64)[1])
    return np.sort(w[WS_HEAD // 4:WS_HEAD // 4 + n])


def workspace(rows: int, stale_row: int):
    """A workspace for `rows` events, filled with int32 `stale_row` (what a hand-out order read past its end finds)."""
    wsb = int(_lib.lib().ct_cusum_workspace_bytes(rows))
    return torch.full(((wsb + 7) // 8 * 2,), stale_row, dtype=torch.int32, device="cuda"), wsb


def outputs(rows: int, ml: int) -> list:
    return [torch.full((rows,), SENT_NL, dtype=torch.int32, device="cuda"),
            torch.empty((rows, ml + 1), dtype=torch.int32, device="cuda"),
            torch.full((rows, ml), SENT_F64, dtype=torch.float64, device="cuda"),
            torch.full((rows, ml), SENT_F64, dtype=torch.float64, device="cuda"),
            torch.full((rows,), SENT_OVF, dtype=torch.uint8, device="cuda")]


def trace(y: np.ndarray, offset: int) -> torch.Tensor:
    buf = torch.zeros(y.size + 16, dtype=torch.float32, device="cuda")
    t = buf[offset:offset + y.size]
    t.copy_(torch.from_numpy(y))
    return t


def launch(y, w0, w1, ty, n, delta, h, ml, out, ws, wsb, count=None):
    """ct_cusum_batch (count None: n events) or ct_cusum_batch_dev (count on the device, capacity n); returns rc."""
    L = _lib.lib()
    d = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).cuda()
    w0, w1, ty = d(w0, np.int64), d(w1, np.int64), d(ty, np.int32)
    st = torch.cuda.current_stream().cuda_stream
    o = [t.data_ptr() for t in out]
    if count is None:
        rc = L.ct_cusum_batch(y.data_ptr(), y.numel(), w0.data_ptr(), w1.data_ptr(), ty.data_ptr(), n, delta, h, ml, *o,
                              ws.data_ptr(), wsb, st)
    else:
        cnt = torch.tensor([count], dtype=torch.int64, device="cuda")
        rc = L.ct_cusum_batch_dev(y.data_ptr(), y.numel(), w0.data_ptr(), w1.data_ptr(), ty.data_ptr(), cnt.data_ptr(), n,
                                  delta, h, ml, *o, ws.data_ptr(), wsb, st)
    torch.cuda.synchronize()
    return rc


def assert_rows(got, want, rows, ml):
    nl, ed, mu, sd, ov = (g[rows] for g in got)
    wnl, wed, wmu, wsd, wov = (w[rows] for w in want)
    assert np.array_equal(nl, wnl), ("n_levels", np.nonzero(nl != wnl)[0][:10])
    assert np.array_equal(ov, wov), ("overflow", np.nonzero(ov != wov)[0][:10])
    assert np.array_equal(ed, wed), ("edges", np.nonzero((ed != wed).any(axis=1))[0][:10])
    used = np.arange(ml)[None, :] < wnl[:, None]
    assert np.array_equal(mu[used], wmu[used]), "mean"
    assert np.array_equal(sd[used], wsd[used]), "std"


def run_case(c: cc.Case, offset: int):
    """Run the case with the trace `offset` floats into an allocation; check which kernel took each window and every
    output against the twin.  Returns the outputs as NumPy arrays."""
    y = trace(c.y, offset)
    assert (y.data_ptr() % 16 == 0, y.data_ptr() % 32 == 0) == (offset % 4 == 0, offset % 8 == 0)
    out = outputs(c.n, c.max_levels)
    ws, wsb = workspace(c.n, c.n - 1)
    _lib.check(launch(y, c.w0, c.w1, c.types, c.n, c.delta, c.h, c.max_levels, out, ws, wsb), "ct_cusum_batch")
    assert np.array_equal(pending_rows(ws), cc.pending(c.y, c.w0, c.w1, c.types, c.n, y.data_ptr() % 16 == 0))
    got = [t.cpu().numpy() for t in out]
    assert_rows(got, cc.twin(c), slice(None), c.max_levels)
    return got


@pytest.mark.parametrize("offset", (0, 1, 4, 8))      # 0, 4, 16, 32 bytes: both kernels aligned, neither, lanes only
@pytest.mark.parametrize("n_events", (cc.SEQ_MIN_EVENTS - 1, cc.SEQ_MIN_EVENTS))
def test_dispatch_boundaries(n_events, offset):
    """Which kernel takes each window at the batch-size, window-length and alignment limits."""
    run_case(cc.dispatch(n_events), offset)


@pytest.mark.parametrize("offset", LANES_AND_WARPS)
@pytest.mark.parametrize("tail", (0, 1, 13, 31))
def test_line_grid_and_trace_end(tail, offset):
    c = cc.line_grid(tail)
    got = run_case(c, offset)
    for i in c.groups["dup"]:
        assert all(np.array_equal(g[i], g[i - 1]) for g in got), i


@pytest.mark.parametrize("offset", LANES_AND_WARPS)
def test_reciprocal_table(offset):
    run_case(cc.recip_table(), offset)


@pytest.mark.parametrize("offset", LANES_AND_WARPS)
@pytest.mark.parametrize("delta,h", [(400.0, 10.0), (400.0, 1000.0), (1e5, 10.0)])
def test_quiet_sum_guard(delta, h, offset):
    run_case(cc.quiet_sum(delta, h), offset)


@pytest.mark.parametrize("offset", LANES_AND_WARPS)
@pytest.mark.parametrize("kind", ("step", "spike"))
def test_increment_clamp(kind, offset):
    run_case(cc.clamp(kind), offset)


@pytest.mark.parametrize("offset", LANES_AND_WARPS)
@pytest.mark.parametrize("max_levels", (2, 3, 4, 32, 33, 64, 1024))
def test_max_levels(max_levels, offset):
    run_case(cc.levels(max_levels), offset)


@pytest.mark.parametrize("offset", LANES_AND_WARPS)
def test_signs_and_domain(offset):
    run_case(cc.domain(), offset)


@pytest.mark.parametrize("offset", LANES_AND_WARPS)
@pytest.mark.parametrize("delta,h", cc.PARAMS)
def test_parameter_limits(delta, h, offset):
    run_case(cc.params(delta, h), offset)


@pytest.mark.parametrize("offset", LANES_AND_WARPS)
def test_rejected_windows(offset):
    c = cc.rejected()
    nl, ed, _, _, ov = run_case(c, offset)
    bad = c.groups["bad"]
    assert np.all(nl[bad] == 0) and np.all(ov[bad] == 0) and np.all(ed[bad] == -1)


@pytest.mark.parametrize("arg,value", [("max_levels", 1), ("max_levels", 1025), ("h", 0.0), ("h", cc.H_MAX + 1),
                                       ("h", float("nan")), ("delta", 0.0), ("delta", -400.0), ("delta", float("nan")),
                                       ("workspace", -8)])
def test_rejected_arguments(arg, value):
    """cusum_launch refuses the call before it touches an output."""
    c = cc.subset(cc.rejected(), np.arange(40))
    kw = dict(delta=400.0, h=10.0, max_levels=16)
    if arg != "workspace":
        kw[arg] = value
    ml = min(max(kw["max_levels"], 2), 1024)
    out = outputs(c.n, ml)
    ws, wsb = workspace(c.n, 0)
    rc = launch(trace(c.y, 0), c.w0, c.w1, c.types, c.n, kw["delta"], kw["h"], kw["max_levels"], out, ws,
                wsb + (value if arg == "workspace" else 0))
    with pytest.raises(ValueError):
        _lib.check(rc, "ct_cusum_batch")
    assert torch.all(out[0] == SENT_NL) and torch.all(out[4] == SENT_OVF)


@pytest.mark.parametrize("count", cc.DEVICE_COUNTS)
def test_device_count_entry(count):
    """ct_cusum_batch_dev as TraceAnalyzer.run calls it: capacity rows, the count in device memory, the workspace and
    the outputs reused from run to run.  Rows below the count equal the twin; the rows at or beyond it (garbage and
    stale windows) keep what they held in n_levels, overflow, mean and std."""
    c = cc.device_rows()
    w0, w1, ty = cc.device_batch(count)
    y = trace(c.y, 0)
    out = outputs(cc.CAPACITY, c.max_levels)
    ws, wsb = workspace(cc.CAPACITY, cc.CAPACITY - 1)
    want = cc.twin(c)
    for _ in range(2):
        _lib.check(launch(y, w0, w1, ty, cc.CAPACITY, c.delta, c.h, c.max_levels, out, ws, wsb, count=count),
                   "ct_cusum_batch_dev")
        assert np.array_equal(pending_rows(ws), cc.pending(c.y, w0, w1, ty, count, True))
        got = [t.cpu().numpy() for t in out]
        assert_rows(got, want, slice(0, count), c.max_levels)
        nl, _, mu, sd, ov = (g[count:] for g in got)
        assert np.all(nl == SENT_NL) and np.all(ov == SENT_OVF) and np.all(mu == SENT_F64) and np.all(sd == SENT_F64)
