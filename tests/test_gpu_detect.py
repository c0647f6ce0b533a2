"""GPU parity: baseline block statistics and threshold/hysteresis detection vs the oracle
definition, on IDENTICAL float32 input (SURVEY.md H2): every integer is bit-exact."""
import numpy as np
import pytest
import torch

from cusumtools_b200 import _lib, detect, filters, synth
from oracle import c_twin, events_oracle as eo

pytestmark = pytest.mark.gpu
S = synth.CHIMERA_SETTINGS


@pytest.fixture(scope="module")
def filtered():
    codes, starts = synth.c1_trace(n=1_000_000, n_events=240, seed=2)
    y = filters.dequant_filtfilt(torch.from_numpy(codes).cuda(), S, 1e5, 8)
    torch.cuda.synchronize()
    return y, starts


@pytest.mark.parametrize("block", [4096, 65536, 1 << 20])
def test_block_stats_exact(filtered, block):
    y, _ = filtered
    bl = detect.baseline_blocks(y, block, 4700.0, 5300.0)
    yh = y.cpu().numpy()
    c0 = np.float32(5000.0)
    shift = eo.stats_shift(300.0, block)
    cnt, s1, s2 = c_twin.block_stats(yh, block, 4700.0, 5300.0, c0, shift)
    assert np.array_equal(bl.count, cnt)
    mean, std = eo.baseline_from_stats(cnt, s1, s2, c0, shift)
    assert np.array_equal(bl.mean, mean) and np.array_equal(bl.std, std)


@pytest.mark.parametrize("block", [4096, 65536])
def test_detection_bit_exact(filtered, block):
    y, true_starts = filtered
    bl = detect.baseline_blocks(y, block, 4700.0, 5300.0).with_thresholds(5.0, 1.0)
    ev = detect.detect_events(y, bl)
    yh = y.cpu().numpy()
    s, e, o = c_twin.detect_events(yh, block, bl.sign, bl.t_start, bl.t_end)
    assert np.array_equal(ev.starts.cpu().numpy(), s)
    assert np.array_equal(ev.ends.cpu().numpy(), e)
    assert ev.open_start == o
    # every injected event is found (the median pad adds one edge artefact at the end)
    got = ev.starts.cpu().numpy()
    assert all(np.any(np.abs(got - t) < 40) for t in true_starts) and len(true_starts) <= len(ev) <= len(true_starts) + 2
    s2, e2, _ = eo.detect_events(yh, block, bl.sign, bl.t_start, bl.t_end)
    assert np.array_equal(s, s2) and np.array_equal(e, e2)


def test_detection_edge_cases():
    block = 4096
    bl = detect.Baseline(block=block, mean=np.array([100.0]), std=np.array([1.0]), count=np.array([1]))
    bl.sign = np.array([1], np.int32); bl.t_start = np.array([90.0], np.float32); bl.t_end = np.array([95.0], np.float32)
    y = np.full(100, 100, np.float32)
    ev = detect.detect_events(torch.from_numpy(y).cuda(), bl)
    assert len(ev) == 0 and ev.open_start == -1
    y[10:20] = 50; y[20] = 92; y[21] = 96; y[90:] = 10
    ev = detect.detect_events(torch.from_numpy(y).cuda(), bl)
    assert ev.starts.tolist() == [10] and ev.ends.tolist() == [21] and ev.open_start == 90
    # starts inside an event
    ev = detect.detect_events(torch.from_numpy(y[15:].copy()).cuda(), bl, state_in=True)
    assert ev.starts.tolist() == [] and ev.open_start == 75
    # tiny capacity forces the retry path
    z = np.full(40000, 100, np.float32); z[::100] = 0
    ev = detect.detect_events(torch.from_numpy(z).cuda(), detect.Baseline(block, np.full(10, 100.0), np.ones(10), np.ones(10, np.int64)).with_thresholds(5.0, 1.0), capacity=7)
    assert len(ev) == 400 and ev.ends.tolist()[:2] == [1, 101]


def test_random_symbol_streams_match_sequential_definition():
    block = 4096
    # end line 95 above the start line 90, and the two lines equal (hysteresis 0): a sample on 90 is then neither symbol
    for t_end, values, p in ((95.0, [80, 92, 100], [0.02, 0.9, 0.08]), (90.0, [80, 90, 92, 100], [0.02, 0.05, 0.85, 0.08])):
        rng = np.random.default_rng(5)
        for n in (1, 31, 32, 33, 4095, 4096, 4097, 100000):
            y = rng.choice(np.array(values, np.float32), size=n, p=p)
            nb = (n + block - 1) // block
            bl = detect.Baseline(block, np.full(nb, 100.0), np.ones(nb), np.ones(nb, np.int64))
            bl.sign = np.ones(nb, np.int32); bl.t_start = np.full(nb, 90, np.float32); bl.t_end = np.full(nb, t_end, np.float32)
            for state_in in (False, True):
                ev = detect.detect_events(torch.from_numpy(y).cuda(), bl, state_in=state_in)
                s, e, o = c_twin.detect_events(y, block, bl.sign, bl.t_start, bl.t_end, state_in=state_in)
                assert ev.starts.tolist() == s.tolist() and ev.ends.tolist() == e.tolist() and ev.open_start == o, (t_end, n)


@pytest.mark.parametrize("block,nb", [(4096, 37), (4096, 2500), (8192, 1)])
def test_blocks_without_baseline_samples_inherit_the_nearest_earlier_valid_block(block, nb):
    """Blocks whose samples all lie outside [baseline_min, baseline_max] (a clogged pore, a long event) take the
    table row of the nearest earlier valid block, leading ones that of the first valid block
    (oracle/events_oracle.py::baseline_from_stats) - many blocks, runs of invalid blocks across thread chunks."""
    rng = np.random.default_rng(block + nb)
    n = block * nb - 17
    y = (5000.0 + rng.normal(0, 20, n)).astype(np.float32)
    bad = rng.random(nb) < 0.4
    bad[0] = nb > 1                                    # leading invalid blocks
    if nb > 40:
        bad[5:30] = True; bad[1000:2100] = True        # long runs
    for k in np.nonzero(bad)[0]:
        y[k * block:(k + 1) * block] -= np.float32(2000.0)
    if nb == 1:
        bad[:] = False
        y[:] = (5000.0 + rng.normal(0, 20, n)).astype(np.float32)
    bl = detect.baseline_blocks(torch.from_numpy(y).cuda(), block, 4700.0, 5300.0, threshold=5.0, hysteresis=1.0)
    c0 = np.float32(5000.0)
    shift = eo.stats_shift(300.0, block)
    cnt, s1, s2 = c_twin.block_stats(y, block, 4700.0, 5300.0, c0, shift)
    mean, std = eo.baseline_from_stats(cnt, s1, s2, c0, shift)
    assert (cnt < 16).sum() == bad.sum()
    assert np.array_equal(bl.mean, mean) and np.array_equal(bl.std, std)
    sign, ts, te = eo.thresholds(mean, std, 5.0, 1.0)
    assert np.array_equal(bl.sign, sign) and np.array_equal(bl.t_start, ts) and np.array_equal(bl.t_end, te)


@pytest.mark.parametrize("hysteresis", [-1.0, -1e-9, float("nan")])
def test_baseline_finalize_rejects_crossed_lines(hysteresis):
    """A negative hysteresis puts the end line beyond the start line, where the detector's definition does not hold:
    ct_baseline_finalize refuses it before any launch and leaves every output as it was.  A NaN threshold (no lines
    wanted) with hysteresis 0 still passes."""
    L = _lib.lib()
    nb = 5
    cnt = torch.full((nb,), 100, dtype=torch.int64, device="cuda")
    s1 = torch.zeros(nb, dtype=torch.int64, device="cuda"); s2 = torch.full((nb,), 400, dtype=torch.int64, device="cuda")
    outs = [torch.full((nb,), -3.0, dtype=torch.float64, device="cuda"), torch.full((nb,), -3.0, dtype=torch.float64, device="cuda"),
            torch.full((nb,), 7, dtype=torch.int32, device="cuda"), torch.full((nb,), -3.0, dtype=torch.float32, device="cuda"),
            torch.full((nb,), -3.0, dtype=torch.float32, device="cuda"), torch.full((1,), 9, dtype=torch.int32, device="cuda")]
    st = torch.cuda.current_stream().cuda_stream
    args = lambda thr, hys: (cnt.data_ptr(), s1.data_ptr(), s2.data_ptr(), nb, 5000.0, 0, 16, thr, hys,
                             *[t.data_ptr() for t in outs], st)
    before = [t.clone() for t in outs]
    assert L.ct_baseline_finalize(*args(5.0, hysteresis)) != 0
    assert "hysteresis" in _lib.lib().ct_last_error().decode()
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(outs, before))
    assert L.ct_baseline_finalize(*args(float("nan"), 0.0)) == 0
    assert L.ct_baseline_finalize(*args(5.0, 0.0)) == 0
    torch.cuda.synchronize()
    assert int(outs[5].item()) == 0 and torch.equal(outs[3], outs[4])


def test_device_table_rejects_negative_hysteresis():
    y = torch.full((1 << 16,), 5000.0, device="cuda")
    bl = detect.baseline_blocks(y, 4096, 4700.0, 5300.0)
    with pytest.raises(ValueError, match="hysteresis"):
        bl.with_thresholds(5.0, -1.0)
    with pytest.raises(ValueError, match="hysteresis"):
        detect.intra_crossings(y, torch.zeros(1, dtype=torch.int64, device="cuda"), torch.ones(1, dtype=torch.int64, device="cuda"),
                               torch.zeros(1, dtype=torch.int64, device="cuda"), bl, 50.0, -5.0)
