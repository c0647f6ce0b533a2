"""CPU: the file-series window gathered into one host buffer equals the reference's slicing
(plot-trace.py:220-270 concatenates the same memmap pieces before scaling)."""
import os

import numpy as np
import scipy.io as sio

from cusumtools_b200 import loader, synth


def _write_series(tmp_path, lengths, seed=0):
    rng = np.random.default_rng(seed)
    parts = []
    for i, n in enumerate(lengths):
        codes = (rng.integers(0, 1 << 14, n).astype(np.uint16) << 2)
        name = os.path.join(tmp_path, f"run_20200101_0000{i:02d}.log")
        codes.tofile(name)
        sio.savemat(name.replace(".log", ".mat"), {k: np.array([[v]]) for k, v in synth.CHIMERA_SETTINGS.items()})
        parts.append(codes)
    return os.path.join(tmp_path, "run_20200101_000000.log"), np.concatenate(parts)


def test_host_codes_spans_files(tmp_path):
    first, allc = _write_series(str(tmp_path), [5000, 7000, 3000])
    s = loader.ChimeraSeries(first)
    assert s.total_samples == 15000 and len(s.sorted_files) == 3
    fs = s.samplerate
    for a, b in ((0, 15000), (100, 4000), (4000, 13000), (5000, 12000), (11999, 15000)):
        host, settings = s.host_codes(a / fs + 1e-9, b / fs + 1e-9)
        assert host.dtype.is_floating_point is False and not host.is_cuda
        lo, hi = int((a / fs + 1e-9) * fs), min(int((b / fs + 1e-9) * fs), 15000)
        assert np.array_equal(host.numpy(), allc[lo:hi])
        assert float(np.squeeze(settings["SETUP_ADCBITS"])) == float(np.squeeze(synth.CHIMERA_SETTINGS["SETUP_ADCBITS"]))


def test_window_reader_reads_ranges_across_files(tmp_path):
    """The streamed loader's source: any sub-range of the window, across file boundaries, straight into caller memory."""
    first, allc = _write_series(str(tmp_path), [5000, 7000, 3000], seed=4)
    s = loader.ChimeraSeries(first)
    fs = s.samplerate
    for a, b in ((0, 15000), (100, 14000), (5000, 12000)):
        rd = s.reader(a / fs + 1e-9, b / fs + 1e-9)
        lo, hi = int((a / fs + 1e-9) * fs), min(int((b / fs + 1e-9) * fs), 15000)
        assert rd.n == hi - lo
        for x, y in ((0, rd.n), (1, 2), (rd.n // 3, 2 * rd.n // 3), (rd.n - 5, rd.n), (4990 - min(lo, 4990), min(rd.n, 5010))):
            if not 0 <= x < y <= rd.n:
                continue
            buf = np.zeros(y - x + 3, np.uint16)
            rd.read_into(buf, x, y)
            assert np.array_equal(buf[:y - x], allc[lo + x:lo + y]) and not buf[y - x:].any()
        rd.close()
    # files of odd lengths; windows inside files at both ends, from a file boundary (an empty first piece) and inside
    # one file; about 200 ranges each: empty ones, single samples, every file boundary crossed, the whole window and
    # random ones.  Nothing past b - a of the destination is written.
    odd = os.path.join(str(tmp_path), "odd")
    os.makedirs(odd)
    first, allc = _write_series(odd, [5001, 7003, 3007], seed=5)
    s = loader.ChimeraSeries(first)
    fs, fsi = s.samplerate, s.file_start_index
    rng = np.random.default_rng(6)
    for a, b in ((101, 14_000), (5001, 14_900), (5100, 11_000)):
        rd = s.reader((a + 0.25) / fs, (b + 0.25) / fs)
        assert rd.n == b - a
        bounds = [int(f) - a for f in fsi if a < f < b]
        ranges = [(0, 0), (rd.n, rd.n), (0, 1), (rd.n - 1, rd.n), (0, rd.n)]
        ranges += [(c, c) for c in bounds] + [(c - 1, c + 1) for c in bounds] + [(c, c + 1) for c in bounds]
        if len(bounds) == 2:
            ranges.append((bounds[0] - 3, bounds[1] + 3))
        while len(ranges) < 200:
            x, y = sorted(rng.integers(0, rd.n + 1, 2))
            ranges.append((int(x), int(y)))
        for x, y in ranges:
            buf = np.full(y - x + 5, 0xA5A5, np.uint16)
            rd.read_into(buf, x, y)
            assert np.array_equal(buf[:y - x], allc[a + x:a + y]), (a, b, x, y)
            assert np.all(buf[y - x:] == 0xA5A5), (a, b, x, y)
        rd.close()
