"""Host logic of the headless entry-point mirrors (cusumtools_b200/app.py): entries, series discovery,
analysis-directory overlays (plot-trace.py:172-203, 350-414) — nothing here launches a kernel."""
import os

import numpy as np
import pandas as pd
import pytest
import scipy.io as sio

from cusumtools_b200 import app as ctapp
from cusumtools_b200 import synth
from oracle import trace_oracle as to


def write_series(tmp_path, n_each=(3000, 5000, 2000)):
    rng = np.random.default_rng(11)
    paths = []
    for i, n in enumerate(n_each):
        name = tmp_path / f"pore_20210305_1015{i:02d}.log"
        ((rng.integers(0, 16384, n).astype(np.uint16)) << 2).astype(np.uint16).tofile(name)
        sio.savemat(str(name).replace(".log", ".mat"), synth.CHIMERA_SETTINGS)
        paths.append(str(name))
    return paths


def test_entry_behaves_like_a_tk_entry():
    e = ctapp.Entry()
    assert e.get() == ""
    e.insert(0, "900000")
    assert e.get() == "900000"
    e.delete(0, "end")
    e.insert("end", "1e5")
    assert e.get() == "1e5"
    v = ctapp.Entry(0)
    v.set(1)
    assert v.get() == 1


def test_app_discovers_the_series_like_the_reference(tmp_path):
    paths = write_series(tmp_path)
    a = ctapp.App(None, paths[2])
    assert a.sorted_files == to.get_filenames(paths[2])
    maps, settings, fsi, total = to.load_memmaps(a.sorted_files)
    assert a.total_samples == total == 10000 and np.array_equal(a.file_start_index, fsi)
    assert a.samplerate == np.floor(np.squeeze(synth.CHIMERA_SETTINGS["ADCSAMPLERATE"]))
    assert a.wildcard.get() == "Found 3 files matching " + paths[2][:-19] + "*.log"
    # GUI defaults of plot-trace.py:100-127
    assert (a.start_entry.get(), a.end_entry.get(), a.cutoff_entry.get(), a.order_entry.get()) == ("0", "10", "900000", "8")
    assert a.psd_length_entry.get() == "" and a.downsample_entry.get() == "" and a.normalize.get() == 0
    assert not (a.events_flag or a.baseline_flag or a.overlay_flag)
    for n in (0, 2999, 3000, 3001, 8000, 8001, 10000):
        assert a.get_file_index(n) == min(to.get_file_index(fsi, n), 2)


def test_missing_series_raises(tmp_path):
    with pytest.raises(FileNotFoundError):
        ctapp.App(None, str(tmp_path / "none_20210305_101500.log"))


def make_analysis_dir(d):
    os.makedirs(d, exist_ok=True)
    pd.DataFrame({"id": [0, 1, 2, 3, 4], "type": [0, 3, 1, 0, 2],
                  "start_time_s": [0.95, 1.10, 1.30, 1.70, 1.95], "end_time_s": [1.02, 1.12, 1.31, 1.72, 2.05]}
                 ).to_csv(os.path.join(d, "rate.csv"), index=False)
    pd.DataFrame({"time_s": [0.0, 0.5, 1.0, 1.5, 2.0], "baseline_pA": [5000.0, 5001.0, -4000.0, 5003.0, 5004.0],
                  "stdev_pA": [20.0, 21.0, 22.0, 23.0, 24.0]}).to_csv(os.path.join(d, "baseline.csv"), index=False)
    with open(os.path.join(d, "summary.txt"), "w") as f:
        f.write("threshold=5.5\nhysteresis=1.25\nintra_threshold=9\nintra_hysteresis=8\ncutoff=100000\npoles=8\n")


def test_overlay_cusum_reads_the_analysis_directory(tmp_path):
    paths = write_series(tmp_path)
    a = ctapp.App(None, paths[0])
    make_analysis_dir(str(tmp_path / "an"))
    a.overlay_cusum(str(tmp_path / "an"))
    assert (a.threshold, a.hysteresis, a.config_cutoff, a.config_order) == (5.5, 1.25, 100000, 8)
    assert a.events_flag and a.baseline_flag and a.overlay_flag
    a.start_time, a.end_time = 1.0, 2.0
    good, bad = a._event_spans()
    # plot-trace.py:353-363: starts and ends selected separately inside [1, 2); a leading end without its
    # start (event 0 ends at 1.02) makes the first start later than the first end -> the reference drops that start
    assert len(good) == 1 and good[0] == pytest.approx((1.70e6, 1.02e6))
    assert len(bad) == 1 and bad[0] == pytest.approx((1.10e6, 1.12e6))
    lines = a._baseline_lines()
    # blocks from the one holding start_time (1.0) up to end_time
    assert [round(l[0]) for l in lines] == [1000000, 1500000] and [round(l[1]) for l in lines] == [1500000, 2000000]
    m, s = -4000.0, 22.0
    assert lines[0][2:] == pytest.approx((m, m + (5.5 - 1.25) * s, m + 5.5 * s))          # negative baseline: lines above it
    m, s = 5003.0, 23.0
    assert lines[1][2:] == pytest.approx((m, m - (5.5 - 1.25) * s, m - 5.5 * s))


def test_overlay_without_rate_file_sets_the_status(tmp_path):
    paths = write_series(tmp_path)
    a = ctapp.App(None, paths[0])
    d = str(tmp_path / "an")
    make_analysis_dir(d)
    os.remove(os.path.join(d, "rate.csv"))
    a.overlay_cusum(d)
    assert not a.overlay_flag and a.wildcard.get() == "rate.csv not found in given directory"


def test_exports_before_plotting_set_the_status(tmp_path):
    paths = write_series(tmp_path)
    a = ctapp.App(None, paths[0])
    a.export_psd(str(tmp_path / "p.csv"))
    assert a.wildcard.get() == "Plot the PSD first"
    a.export_trace(str(tmp_path / "t.csv"))
    assert a.wildcard.get() == "Plot the trace first"
    assert not os.path.exists(tmp_path / "p.csv")


def test_fit_helpers_match_the_reference_formulas():
    a = ctapp.App.__new__(ctapp.App)
    f = np.array([1.0, 10.0, 100.0])
    assert np.allclose(a.fitfunc(f, 2.0, 1.5, 30.0, 0.01),
                       np.log10((2.0 / f) ** 1.5 + 1.5 * (2.0 / 30.0) ** 2.5 * (f / 2.0) + 0.01))
    assert np.isclose(a.old_L(np.array([1.0, 3.0]), 0.5, 2.0), 1.0)
    assert np.isclose(ctapp.psd_fit(10.0, 1e-3, 1.0, 1e-3), np.log10(1e-2 + 1 + 1e-4))


def test_overlay_cusum_agrees_with_the_live_reference(tmp_path):
    """plot-trace.py:172-203 run headlessly on the same analysis directory (when CUSUMTOOLS_REFERENCE names a
    cusumtools checkout)."""
    from types import SimpleNamespace
    from oracle import reference_shim as ref
    if not ref.available():
        pytest.skip("CUSUMTOOLS_REFERENCE does not name a cusumtools checkout")
    pt = ref.load("plot-trace.py")
    d = str(tmp_path / "an")
    make_analysis_dir(d)
    pt.tkinter.filedialog.askdirectory = lambda **k: d
    r = SimpleNamespace(wildcard=ctapp.Entry())
    pt.App.overlay_cusum(r)
    a = ctapp.App(None, write_series(tmp_path)[0])
    a.overlay_cusum(d)
    for k in ("threshold", "hysteresis", "config_cutoff", "config_order", "events_flag", "baseline_flag", "overlay_flag"):
        assert getattr(a, k) == getattr(r, k), k
    assert a.ratefile.equals(r.ratefile) and a.baseline_file.equals(r.baseline_file)
