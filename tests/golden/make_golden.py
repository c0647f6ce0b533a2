"""Generates tests/golden/*.npz by running the REFERENCE'S OWN code headlessly
(plot-trace.py and noise-fit.py of a cusumtools checkout, through oracle/reference_shim.py):
    CUSUMTOOLS_REFERENCE=<cusumtools checkout> python tests/golden/make_golden.py
The fixtures pin oracle/trace_oracle.py (and, through it, the CUDA path) to outputs of the
reference itself; the reference ships no tests or golden vectors of its own.
Library versions used are recorded inside the fixture.
"""
import os
import sys
import tempfile

import numpy as np
import scipy
import scipy.io as sio

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import reference_shim as ref  # noqa: E402
from cusumtools_b200 import synth  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def savez_lzma(path, **arrays):
    """np.savez with LZMA members (np.load reads them as it reads any .npz): noisy float64 traces deflate poorly,
    and a fixture stays under 1 MB."""
    import zipfile
    with zipfile.ZipFile(path, "w", zipfile.ZIP_LZMA) as z:
        for k, v in arrays.items():
            with z.open(k + ".npy", "w", force_zip64=True) as f:
                np.lib.format.write_array(f, np.asanyarray(v), allow_pickle=False)


def edge_fixture():
    """fixture 5: the odd-extension boundary mode of legacy/bessel-filter.py:124-131 on the tool's own 26-sample
    step (generate_step) and on a 3 000-sample noisy step, orders 2 / 4 / 8."""
    rng = np.random.default_rng(7)
    step = np.zeros(26)
    step[13:] = 1.0
    noisy = np.concatenate((np.zeros(1500), np.ones(1500))) + 0.05 * rng.standard_normal(3000)
    out = {"step": step, "noisy": noisy, "fc_khz": 100.0, "fs_khz": 1000.0,
           "versions": np.array([np.__version__, scipy.__version__])}
    for poles in (2, 4, 8):
        out[f"step_{poles}"] = ref.ref_filter_data_edge(step, 100.0, 1000.0, poles)
        out[f"noisy_{poles}"] = ref.ref_filter_data_edge(noisy, 100.0, 1000.0, poles)
    np.savez_compressed(os.path.join(HERE, "edge_fixture.npz"), **out)


def main():
    assert ref.available(), "set CUSUMTOOLS_REFERENCE to a cusumtools checkout"
    if "--only-edge" in sys.argv:
        edge_fixture()
        return
    edge_fixture()
    rng = np.random.default_rng(42)
    settings = synth.CHIMERA_SETTINGS
    fs = np.floor(np.squeeze(settings["ADCSAMPLERATE"]))

    # ---- fixture 1: scale_raw_data + filter_data on a 24 001-sample trace with 5 events
    n = 24001
    cur = 5000 + 150 * rng.standard_normal(n)
    for k in range(5):
        s = 1500 + 4000 * k
        cur[s:s + 1000] -= 800
        cur[s + 1000:s + 2000] -= 1600
    codes = synth.quantise(cur, settings)
    codes[7] |= 3          # dirty low bits: the bitmask must clear them
    data = ref.ref_scale_raw_data(codes, settings, fs)
    out = {"codes": codes, "scaled": data, "fs": fs,
           "versions": np.array([np.__version__, scipy.__version__])}
    for cutoff, order in ((100000, 8), (250000, 8), (900000, 8), (100000, 4), (200000, 5)):
        out[f"filt_{cutoff}_{order}"] = ref.ref_filter_data(data, fs, cutoff, order)
    # even-length variant (median = mean of the two middle values)
    out["filt_even_100000_8"] = ref.ref_filter_data(data[:-1], fs, 100000, 8)
    savez_lzma(os.path.join(HERE, "filter_fixture.npz"), **out)

    # ---- fixture 2: integrate_noise and the welch call as update_psd issues it
    from scipy.signal import welch
    x = ref.ref_filter_data(data, fs, 100000, 8)
    L = 2 ** 12
    f, P = welch(x, fs, nperseg=np.minimum(L, len(x)))          # plot-trace.py:437,442
    rms = ref.ref_integrate_noise(f, P)
    np.savez_compressed(os.path.join(HERE, "psd_fixture.npz"), x=x, fs=fs, nperseg=L, f=f, Pxx=P, rms=rms)

    # ---- fixture 3: file series through get_filenames/load_memmaps/load_mapped_data
    with tempfile.TemporaryDirectory() as d:
        parts = [codes[:9000], codes[9000:15000], codes[15000:]]
        stamps = ["20200101_000002", "20200101_000000", "20200101_000001"]   # unsorted on purpose
        order = np.argsort(stamps)
        pieces = [None] * 3
        for rank, idx in enumerate(order):
            pieces[idx] = parts[rank]
        gains = [1.305, 1.305, 1.305]
        for p, s, g in zip(pieces, stamps, gains):
            base = os.path.join(d, "trace_" + s)
            p.tofile(base + ".log")
            st = dict(settings); st["SETUP_preADCgain"] = np.array([[g]])
            sio.savemat(base + ".mat", st)
        first = os.path.join(d, "trace_" + stamps[0] + ".log")
        w, fs2 = ref.ref_load_mapped_data(first, 0.0005, 0.005)
        np.savez_compressed(os.path.join(HERE, "loader_fixture.npz"), codes=codes, window=w, fs=fs2,
                            start_s=0.0005, end_s=0.005, split=np.array([9000, 15000]))

    # ---- fixture 4: noise-fit SpectrumSample on a synthetic big-endian .bin
    with tempfile.TemporaryDirectory() as d:
        m = 40000
        raw = (1000 + 30 * rng.standard_normal(m))
        rec = np.zeros(m, dtype=np.dtype([("curr_pA", ">f8"), ("volt_mV", ">f8")]))
        rec["curr_pA"] = raw
        rec["volt_mV"] = 200.0
        path = os.path.join(d, "B0001.bin")
        rec.tofile(path)
        s = ref.ref_spectrum_sample(path, 500000, 2 ** np.ceil(np.log2(8192)), 100000)
        np.savez_compressed(os.path.join(HERE, "spectrum_fixture.npz"), raw=raw, fs=500000, psdlength=8192,
                            cutoff=100000, f=s.f, Pxx=s.Pxx, current=s.current)
    print("golden fixtures written to", HERE)


if __name__ == "__main__":
    main()
