"""World-size-2 gloo tests (CPU) of the host-side multi-GPU logic: the global median search
over all-reduced histograms / window counters, global event ids, the shard bounds and the
PSD reduction.  The device kernels are replaced by numpy stand-ins with the same contract
(the GPU tests check the kernels themselves); everything else is the production code."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from cusumtools_b200 import median, pipeline, psd


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, fn, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        out[rank] = fn(rank, world, dist.group.WORLD)
    finally:
        dist.destroy_process_group()


def run2(fn, world=2):
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), fn, out), nprocs=world, join=True)
    return [out[r] for r in range(world)]


def _codes(seed, n):
    rng = np.random.default_rng(seed)
    return ((np.clip(40900 + 64 * rng.standard_normal(n), 0, 65535)).astype(np.uint16) & 0xFFFC).astype(np.uint16)


def _median_job(rank, world, group):
    n_total = 9_000_001                       # odd; > 2^22 so the sampled path + window search runs
    lo, hi = pipeline.shard_bounds(n_total, world, rank, 4096)
    codes = _codes(0, n_total)[lo:hi]
    mask = 0xFFFC

    def hist_fn(stride):
        return torch.from_numpy(np.bincount(codes[::stride] & mask, minlength=65536).astype(np.int32))

    def count_fn(lo_, step):
        c = (codes & mask).astype(np.int64)
        out = [np.sum(c < lo_)] + [np.sum(c == lo_ + i * step) for i in range(8)]
        return torch.tensor(out, dtype=torch.int64)

    return median.search(len(codes), mask, hist_fn, count_fn, group)


def _drift_job(rank, world, group):
    """The estimate comes from a piece that sits 300 codes away from the global median (a drifting trace seen
    through its first seconds): one re-estimate from all the data must put the window right."""
    n_total = 9_000_001
    lo, hi = pipeline.shard_bounds(n_total, world, rank, 4096)
    codes = _codes(0, n_total)[lo:hi]
    mask = 0xFFFC
    calls = {"count": 0}

    def hist_fn(stride):
        return torch.from_numpy(np.bincount(codes[::stride] & mask, minlength=65536).astype(np.int32))

    def first_piece_hist(stride):
        return torch.from_numpy(np.bincount((codes[:100_000:stride] + 300) & mask, minlength=65536).astype(np.int32))

    def count_fn(lo_, step):
        calls["count"] += 1
        c = (codes & mask).astype(np.int64)
        return torch.tensor([np.sum(c < lo_)] + [np.sum(c == lo_ + i * step) for i in range(8)], dtype=torch.int64)

    plan = median.estimate(len(codes), mask, first_piece_hist, group, n_sampled=100_000)
    pair = median.search(len(codes), mask, hist_fn, count_fn, group, plan=plan)
    return pair, calls["count"]


def test_a_poor_first_estimate_costs_one_re_estimate():
    got = run2(_drift_job)
    allc = np.sort(_codes(0, 9_000_001) & 0xFFFC)
    want = (int(allc[(allc.size - 1) // 2]), int(allc[allc.size // 2]))
    assert got[0][0] == want and got[1][0] == want
    assert got[0][1] <= 3                               # the missed window, the re-estimated one (+ at most one step)


def test_global_median_matches_numpy_on_two_ranks():
    got = run2(_median_job)
    allc = np.sort(_codes(0, 9_000_001) & 0xFFFC)
    want = (int(allc[(allc.size - 1) // 2]), int(allc[allc.size // 2]))
    assert got[0] == want and got[1] == want


def _ids_job(rank, world, group):
    return pipeline.event_id_offsets(100 + 7 * rank, group)


def test_event_ids_follow_rank_order():
    assert run2(_ids_job) == [(0, 207), (100, 207)]
    assert run2(_ids_job, world=3) == [(0, 321), (100, 321), (207, 321)]


def _status_job(rank, world, group):
    return pipeline.event_ids_and_status(10 + rank, int(rank == 1), group)


def test_error_status_reaches_every_rank():
    """A rank that failed passes a flag INSTEAD of raising before the collective: every rank sees it in the same
    all_reduce that carries the event counts and takes the same decision (ADVICE r1: no rank left in a collective)."""
    assert run2(_status_job) == [(0, 21, 1), (10, 21, 1)]
    assert pipeline.event_ids_and_status(7, 0) == (0, 7, 0)


def test_shard_bounds_cover_the_trace_and_align():
    for n, world, align in ((2_499_999_600, 8, 1 << 20), (10_000, 3, 4096), (4096 * 5 + 1, 2, 4096)):
        b = [pipeline.shard_bounds(n, world, r, align) for r in range(world)]
        assert b[0][0] == 0 and b[-1][1] == n
        assert all(b[i][1] == b[i + 1][0] for i in range(world - 1))
        assert all(lo % align == 0 for lo, _ in b)


def _psd_job(rank, world, group):
    L, fs = 1024, 4166666.0
    rng = np.random.default_rng(3)
    x = (5000 + 30 * rng.standard_normal(40_000)).astype(np.float32)
    s0, s1, a, b = psd.segment_share(x.size, L, world, rank)
    # numpy stand-in for ct_welch_f32 on this rank's samples: the same raw periodogram sums
    xs = x[a:b].astype(np.float64)
    w = 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(L) / L)
    acc = np.zeros(L // 2 + 1)
    for s in range(s1 - s0):
        seg = xs[s * (L // 2):s * (L // 2) + L]
        acc += np.abs(np.fft.rfft(w * (seg - seg.mean()))) ** 2
    a_sum, nseg = psd.reduce_sums(torch.from_numpy(acc), s1 - s0, group)
    f, P = psd.scale_sums(a_sum, nseg, fs, L)
    return nseg, P


def test_psd_reduction_equals_scipy_welch():
    from scipy.signal import welch
    res = run2(_psd_job)
    rng = np.random.default_rng(3)
    x = (5000 + 30 * rng.standard_normal(40_000)).astype(np.float32)
    f, want = welch(x.astype(np.float64), 4166666.0, nperseg=1024)
    for nseg, P in res:
        assert nseg == (x.size - 512) // 512
        assert np.allclose(P, want, rtol=1e-10, atol=0)


def test_segment_share_partitions_scipys_segments():
    for n, L, world in ((2_499_999_600, 1 << 20, 8), (40_000, 1024, 3), (1000, 1024, 2)):
        nseg = max(0, (n - L // 2) // (L // 2))
        sh = [psd.segment_share(n, L, world, r) for r in range(world)]
        assert sum(s1 - s0 for s0, s1, _, _ in sh) == nseg
        assert all(b <= n for _, _, _, b in sh)


def _gather_job(rank, world, group):
    n = 5 + 3 * rank
    tabs = {"starts": torch.arange(n, dtype=torch.int64) + 1000 * rank, "mean": torch.full((n, 4), float(rank))}
    got = pipeline.gather_tables(tabs, group, dst=0)
    return None if got is None else {k: v.numpy() for k, v in got.items()}


def test_event_tables_are_gathered_in_rank_order():
    res = run2(_gather_job, world=3)
    assert res[1] is None and res[2] is None
    want = np.concatenate([np.arange(5 + 3 * r) + 1000 * r for r in range(3)])
    assert np.array_equal(res[0]["starts"], want)
    assert res[0]["mean"].shape == (want.size, 4) and np.array_equal(res[0]["mean"][:, 0], np.repeat([0.0, 1.0, 2.0], [5, 8, 11]))


def test_standard_error_of_the_estimate_follows_the_density_at_the_median():
    """MedianPlan.se = sqrt(samples) / (2 x samples at the estimate), in code steps: small for a trace that sits on its
    baseline, large when the median falls where few samples are (a drifting baseline; the tail between two levels) -
    what decides between the device-verified window and the host loop (median.route)."""
    rng = np.random.default_rng(5)
    n, mask = 4_000_000, 0xFFFC

    def plan_for(codes):
        def hist_fn(stride):
            return torch.from_numpy(np.bincount(codes[::stride] & mask, minlength=65536).astype(np.int32))
        return median.estimate(len(codes), mask, hist_fn)

    quiet = _codes(1, n)
    p = plan_for(quiet)
    true = int(np.sort(quiet & mask)[(n - 1) // 2])
    assert p.se < 0.1 and abs(p.est - true) <= 4 and p.est % 4 == 0 and p.lo == p.est - 12
    drift = ((quiet.astype(np.int64) + 4 * (np.arange(n) * 3000 // n)) & 0xFFFF).astype(np.uint16)
    assert plan_for(drift).se > 0.8
    # half the samples 340 codes lower (inside events): the median lies in the lower tail of the baseline cluster
    two = quiet.copy()
    two[: int(0.493 * n)] -= np.uint16(4 * 340)
    rng.shuffle(two)
    assert 0.25 < plan_for(two).se < 0.8
    small = _codes(2, 100_000)                              # below 2^20 samples: the full histogram is exact
    ps = plan_for(small)
    srt = np.sort(small & mask)
    assert ps.exact == (int(srt[(len(small) - 1) // 2]), int(srt[len(small) // 2]))
