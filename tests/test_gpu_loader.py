"""GPU parity of the loaders against the oracle restatement of the reference's loaders
(plot-trace.py:220-307, print_trace.py:32-39, legacy/minimal_psd.py:188-193) on files written
in the reference's formats, and of the float median behind np.pad(mode='median')."""
import os

import numpy as np
import pytest
import scipy.io as sio
import torch

from cusumtools_b200 import filters, loader, synth
from oracle import trace_oracle as to

pytestmark = pytest.mark.gpu


def write_series(tmp_path, gains, n_each=50_000, seed=5):
    rng = np.random.default_rng(seed)
    paths = []
    for i, g in enumerate(gains):
        name = tmp_path / f"run_201901{10 + i:02d}_1200{i:02d}.log"
        codes = (rng.integers(0, 16384, n_each).astype(np.uint16) << 2).astype(np.uint16)
        codes.tofile(name)
        st = dict(synth.CHIMERA_SETTINGS)
        st["SETUP_TIAgain"] = g
        sio.savemat(str(name).replace(".log", ".mat"), st)
        paths.append(str(name))
    return paths


def test_chimera_series_single_gain_codes(tmp_path):
    paths = write_series(tmp_path, [100e6, 100e6, 100e6])
    s = loader.ChimeraSeries(paths[1])
    assert [os.path.basename(p) for p in s.sorted_files] == [os.path.basename(p) for p in to.get_filenames(paths[1])]
    fs = s.samplerate
    for t0, t1 in ((0.0, 0.005), (0.010, 0.030), (0.0119, 0.0121), (0.02, 1.0)):
        raw, settings = s.load_codes(t0, t1)
        want = to.load_mapped_data(paths[0], t0, t1)[0]
        got = filters.scale_codes_host(raw.cpu().numpy(), settings)
        assert np.array_equal(got, want)


def test_chimera_series_mixed_gain_pA(tmp_path):
    paths = write_series(tmp_path, [100e6, 50e6, 100e6])
    s = loader.ChimeraSeries(paths[0])
    with pytest.raises(ValueError):
        s.load_codes(0.0, 0.03)
    got = s.load_pA(0.005, 0.030).cpu().numpy()
    want = to.load_mapped_data(paths[0], 0.005, 0.030)[0]
    assert got.shape == want.shape
    w32 = want.astype(np.float32)                            # float64 affine rounded once
    assert np.all(np.abs(got - w32) <= np.spacing(np.abs(w32)))
    assert np.mean(got == w32) > 0.9999


def _special_float64() -> np.ndarray:
    """float64 values where a conversion to float32 goes wrong first: signed zeros, infinities and NaNs, float64
    subnormals, magnitudes at and past the float32 maximum (below the halfway point to 2^128 they round to the maximum,
    from it on to infinity), values that round into the float32 subnormals or to zero, and exact float32 halfway points
    (ties to even) among the normals and the subnormals; then random bit patterns."""
    f32max, tiny = float(np.finfo(np.float32).max), 2.0 ** -149
    half_ulp_max = 2.0 ** 103                                   # half an ulp of the float32 maximum
    v = [0.0, -0.0, np.inf, -np.inf, np.nan, -np.nan, 5e-324, -5e-324, 2.2250738585072009e-308, -1e-310,
         f32max, -f32max, f32max + half_ulp_max * (1 - 2.0 ** -20), f32max + half_ulp_max, -(f32max + half_ulp_max),
         3.5e38, 1e39, -1e300, 1.7976931348623157e308,
         2.0 ** -126, 2.0 ** -126 * (1 - 2.0 ** -24), 1e-40, -3e-42, tiny, 0.5 * tiny, -0.5 * tiny, 0.75 * tiny, 1.5 * tiny,
         2.5 * tiny, -2.5 * tiny, 0.49 * tiny, 1e-46,
         1 + 2.0 ** -24, 1 + 3 * 2.0 ** -24, -(1 + 2.0 ** -24), 2.0 ** 100 * (1 + 2.0 ** -24), 16777217.0, 16777219.0,
         5000 + 2.0 ** -12, -(5000 + 3 * 2.0 ** -12)]
    bits = np.random.default_rng(11).integers(0, 2 ** 64, 4096, dtype=np.uint64)
    return np.concatenate((np.array(v, np.float64), bits.view(np.float64)))


def test_bin_and_legacy_records(tmp_path):
    rng = np.random.default_rng(1)
    n = 30_001
    rec = np.zeros(n, dtype=np.dtype([("curr_pA", ">f8"), ("volt_mV", ">f8")]))
    rec["curr_pA"] = 5000 + 100 * rng.standard_normal(n)
    rec["volt_mV"] = 200.0
    p = tmp_path / "trace.bin"
    rec.tofile(p)
    got = loader.load_bin(str(p), 0.001, 0.004, 4166666.0).cpu().numpy()
    want = to.load_bin(str(p), 0.001, 0.004, 4166666.0)
    assert np.array_equal(got, want.astype(np.float32))
    assert np.array_equal(loader.load_bin(str(p)).cpu().numpy(), rec["curr_pA"].astype(np.float32))
    # .bin currents at the float32 limits: each float64 rounded once to nearest even, subnormals kept, bit for bit what
    # numpy's astype gives (a NaN for a NaN)
    x = _special_float64()
    rec = np.zeros(x.size, dtype=rec.dtype)
    rec["curr_pA"], rec["volt_mV"] = x, -x[::-1]
    rec.tofile(p)
    got = loader.load_bin(str(p)).cpu().numpy()
    with np.errstate(over="ignore"):
        want = x.astype(np.float32)
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan)
    assert np.array_equal(got[~nan].view(np.uint32), want[~nan].view(np.uint32))
    sub = (want != 0) & (np.abs(want) < np.finfo(np.float32).tiny)
    assert (want.view(np.uint32) == 0x80000000).any() and np.isinf(want).sum() >= 4 and sub.sum() >= 8
    # legacy records
    leg = np.zeros(n, dtype=np.dtype([("current", ">i2"), ("voltage", ">i2")]))
    leg["current"] = rng.integers(-32768, 32767, n)
    leg["voltage"] = 7
    q = tmp_path / "legacy.dat"
    leg.tofile(q)
    got = loader.load_legacy_i2(str(q), 100, 20_000, 0.25).cpu().numpy()
    want = to.load_legacy_i2(str(q), 100, 20_000, 0.25)
    assert np.array_equal(got, want.astype(np.float32))
    # every int16 value, shuffled, then an odd tail: savegain * current is a float64 product in the reference, so the
    # float32 result is that product rounded once (a float32 gain times a float32 value is one ulp off for many gains)
    m = 65536 + 1001
    leg = np.zeros(m, dtype=leg.dtype)
    leg["current"][:65536] = rng.permutation(np.arange(-32768, 32768, dtype=np.int16))
    leg["current"][65536:] = rng.integers(-32768, 32768, m - 65536)
    leg["voltage"] = rng.integers(-32768, 32768, m)
    leg.tofile(q)
    for gain in (0.25, 0.1, 1 / 3, 2.5e-3, 20 / 32768):
        for a, b in ((0, m), (7, m - 2)):
            got = loader.load_legacy_i2(str(q), a, b, gain).cpu().numpy()
            assert np.array_equal(got, to.load_legacy_i2(str(q), a, b, gain).astype(np.float32)), (gain, a, b)


@pytest.mark.parametrize("n", [1, 2, 1001, 1002, 300_000])
def test_float_median_exact(n):
    rng = np.random.default_rng(n)
    x = (5000 + 150 * rng.standard_normal(n)).astype(np.float32)
    x[rng.integers(0, n, max(1, n // 10))] *= -1
    t = torch.from_numpy(x).cuda()
    assert filters.float_median(t) == float(np.median(x.astype(np.float64)))
    assert filters.float_median(t, use_abs=True) == float(np.median(np.abs(x).astype(np.float64)))


def test_filter_data_on_bin_trace_takes_the_median_pad(tmp_path):
    rng = np.random.default_rng(2)
    x = (5000 + 150 * rng.standard_normal(200_000)).astype(np.float32)
    x[50_000:52_000] -= 800
    y = filters.bessel_filtfilt(torch.from_numpy(x).cuda(), 4166666.0, 1e5, 8).cpu().numpy()
    want = to.filter_data(x.astype(np.float64), 4166666.0, 1e5, 8)
    assert np.abs(y - want).max() < 0.05


# A three-file `.log` series of odd lengths, and windows of it in samples: one that starts and ends inside files, one
# that starts exactly on a file boundary (its first piece is empty: plot-trace.py:220-227 picks the earlier file) and
# one inside a single file.
FILE_LENGTHS = (1_100_003, 900_001, 1_000_007)
STAMPS = ("20210301_120000", "20210301_120001", "20210301_120002")
WINDOWS = {"mid_to_mid": (100_003, 2_900_001), "on_boundary": (1_100_003, 2_950_001), "one_file": (1_150_001, 1_990_001)}
STREAM_KW = dict(threshold=5.0, hysteresis=1.0, baseline_block=65536, baseline_min=4700.0, baseline_max=5300.0,
                 cusum_delta=400.0, cusum_h=10.0)


def write_pore_series(d, codes) -> list:
    cuts = np.concatenate(([0], np.cumsum(FILE_LENGTHS)))
    assert cuts[-1] == codes.size
    files = []
    for i, st in enumerate(STAMPS):
        base = os.path.join(str(d), "pore_" + st)
        codes[cuts[i]:cuts[i + 1]].tofile(base + ".log")
        sio.savemat(base + ".mat", synth.CHIMERA_SETTINGS)
        files.append(base + ".log")
    return files


def file_codes(files) -> np.ndarray:
    """The series' codes read independently of the loader."""
    return np.concatenate([np.fromfile(f, dtype=np.uint16) for f in files])


def window_reader(files, window):
    """(reader, first sample, last sample + 1) of a window given in samples."""
    a, b = WINDOWS[window] if isinstance(window, str) else window
    series = loader.ChimeraSeries(files[1])
    fs = series.samplerate
    rd = series.reader((a + 0.25) / fs, (b + 0.25) / fs)
    assert rd.n == b - a
    return rd, a, b


@pytest.fixture(scope="module")
def pore_files(tmp_path_factory):
    codes, _ = synth.c1_trace(n=sum(FILE_LENGTHS), n_events=740, seed=21)
    return write_pore_series(tmp_path_factory.mktemp("pore"), codes)


def test_streaming_from_file_equals_streaming_from_host(pore_files):
    """plot-trace.py:230-299 reads the window of a multi-file `.log` series before anything else happens; here the
    files are read piece by piece on a worker thread into rotating pinned slabs while earlier pieces are already
    being copied and analysed.  On each window, with (reader threads, slabs) = (1, 1), (3, 2) and (8, 3): more pieces
    than slabs (with one slab every piece waits for the previous copy), one to eight reader threads per piece.  Same
    sub-shards, same kernels: the result equals the run from one host buffer of the same codes, bit for bit."""
    from cusumtools_b200 import pipeline
    from test_gpu_analyzer_steps import same, stream_snapshot
    codes = file_codes(pore_files)
    for window in WINDOWS:
        rd, a, b = window_reader(pore_files, window)
        if window == "on_boundary":
            assert a == FILE_LENGTHS[0] and rd.spans[0][3] == 0 and len(rd.spans) == 3
        if window == "one_file":
            assert len(rd.spans) == 1
        host = torch.from_numpy(codes[a:b].copy()).pin_memory()
        for threads, slabs in ((1, 1), (3, 2), (8, 3)):
            what = (window, threads, slabs)
            an = pipeline.StreamingAnalyzer(rd.n, rd.settings, 1e5, 8, shards=16, **STREAM_KW)
            assert len(an.sub) > 2 * slabs, what
            from_file = stream_snapshot(an.run_from_file(rd, threads=threads, slabs=slabs))
            from_host = stream_snapshot(an.run_from_host(host))
            assert from_host["scalars"][1] > 0.95 * (b - a) / synth.EVENT_PERIOD, what
            same(from_file, from_host, what)
        rd.close()


def test_file_feed_falls_back_to_the_whole_trace(tmp_path):
    """A sub-shard without a single baseline sample, halos included, sends the streamed run to the whole-trace
    analyzer, which reads the whole window through the file feed: the result equals the run from host memory."""
    from cusumtools_b200 import pipeline
    from test_gpu_analyzer_steps import same, stream_snapshot
    a, b = WINDOWS["mid_to_mid"]
    an = pipeline.StreamingAnalyzer(b - a, synth.CHIMERA_SETTINGS, 1e5, 8, shards=16, **STREAM_KW)
    codes, _ = synth.c1_trace(n=sum(FILE_LENGTHS), n_events=740, seed=22)
    _, _, ea, eb = an.sub[5]
    codes[a + ea:a + eb] += np.uint16(4096)                 # +2.4 nA: no sample inside [baseline_min, baseline_max]
    files = write_pore_series(tmp_path, codes)
    rd, _, _ = window_reader(files, "mid_to_mid")
    got = stream_snapshot(an.run_from_file(rd, threads=3, slabs=2))
    assert got["scalars"][4] == "whole"
    fresh = pipeline.StreamingAnalyzer(b - a, synth.CHIMERA_SETTINGS, 1e5, 8, shards=16, **STREAM_KW)
    same(got, stream_snapshot(fresh.run_from_host(torch.from_numpy(codes[a:b].copy()).pin_memory())), "whole")


def test_a_failing_read_surfaces_and_leaves_the_analyzer_usable(pore_files):
    """A read that comes up short on the reader thread (the last span claims samples past the end of its file) is
    raised by run_from_file as OSError once the thread and its readers have ended; the analyzer's next run equals a
    fresh analyzer's."""
    import threading
    from cusumtools_b200 import pipeline
    from test_gpu_analyzer_steps import same, stream_snapshot
    rd, a, b = window_reader(pore_files, "mid_to_mid")
    off, path, first, cnt = rd.spans[-1]
    held = os.path.getsize(path) // 2
    assert first + cnt <= held
    bad = loader.WindowReader(rd.spans[:-1] + [(off, path, held - cnt + 5000, cnt)], rd.n, rd.settings)
    an = pipeline.StreamingAnalyzer(rd.n, rd.settings, 1e5, 8, shards=16, **STREAM_KW)
    before = threading.active_count()
    with pytest.raises(OSError, match="short read"):
        an.run_from_file(bad, threads=3, slabs=2)
    assert threading.active_count() == before
    bad.close()
    host = torch.from_numpy(file_codes(pore_files)[a:b].copy()).pin_memory()
    got = stream_snapshot(an.run_from_host(host))
    fresh = pipeline.StreamingAnalyzer(rd.n, rd.settings, 1e5, 8, shards=16, **STREAM_KW)
    same(got, stream_snapshot(fresh.run_from_host(host)), "after a failed read")
