"""TEST INFRASTRUCTURE — CPU restatement of stages 1 and 4 of the reference hot path.

Every function follows a reference call sequence line by line; the arithmetic itself is
in numpy/scipy exactly as in the reference (third-party, unpinned: numpy 2.3.5 /
scipy 1.18.1 here).  Pinned against the reference's own code by
tests/test_oracle_pins.py (golden vectors in tests/golden/ + live comparison through
oracle/reference_shim.py whenever CUSUMTOOLS_REFERENCE names a cusumtools checkout).
"""
from __future__ import annotations

import glob
import os
import time

import numpy as np
import scipy.io as sio
from scipy.signal import bessel, filtfilt, lfilter, lfilter_zi, welch

CHIMERA_KEYS = ("ADCSAMPLERATE", "SETUP_TIAgain", "SETUP_preADCgain", "SETUP_pAoffset",
                "SETUP_mVoffset", "SETUP_ADCVREF", "SETUP_ADCBITS")


# ----------------------------------------------------------------------------- loaders
def get_filenames(initialfile: str) -> list[str]:
    """plot-trace.py:301-307 — series discovery by the 19-char timestamp suffix."""
    pattern = initialfile[:-19] + "*.log"
    files = glob.glob(pattern)
    timelist = [os.path.basename(f)[-19:-4] for f in files]
    stamps = [time.mktime(time.strptime(s, "%Y%m%d_%H%M%S")) for s in timelist]
    return [f for (_, f) in sorted(zip(stamps, files), key=lambda p: p[0])]


def load_memmaps(sorted_files):
    """plot-trace.py:289-299."""
    columntypes = np.dtype([("current", np.uint16)])
    maps = [np.memmap(str(f), dtype=columntypes, mode="r")["current"] for f in sorted_files]
    settings = [sio.loadmat(f.replace(".log", ".mat")) for f in sorted_files]
    file_start_index = [0]
    total = 0
    for m in maps:
        total += len(m)
        file_start_index.append(total)
    return maps, settings, np.array(file_start_index, dtype=np.int64), total


def get_file_index(file_start_index, samplenum):
    """plot-trace.py:220-227 (including its out-of-range return on IndexError)."""
    i = 0
    try:
        while file_start_index[i + 1] < samplenum:
            i += 1
    except IndexError:
        i = len(file_start_index)
    return i


def scale_raw_data(tempdata, settings):
    """plot-trace.py:272-287 — uint16 ADC codes -> pA (float64)."""
    TIAgain = np.squeeze(settings["SETUP_TIAgain"])
    preADCgain = np.squeeze(settings["SETUP_preADCgain"])
    currentoffset = np.squeeze(settings["SETUP_pAoffset"])
    ADCvref = np.squeeze(settings["SETUP_ADCVREF"])
    ADCbits = np.squeeze(settings["SETUP_ADCBITS"])
    closedloop_gain = TIAgain * preADCgain
    bitmask = (2 ** 16 - 1) - (2 ** (16 - ADCbits) - 1)
    tempdata = tempdata.astype(np.uint16) & bitmask
    tempdata = ADCvref - (2 * ADCvref) * tempdata.astype(float) / float(2 ** 16)
    tempdata = -tempdata / float(closedloop_gain) + float(currentoffset)
    return tempdata * 1e12


def load_mapped_data(initialfile, start_s, end_s):
    """plot-trace.py:230-270 + 325-327: time window -> one float64 pA vector."""
    files = get_filenames(initialfile)
    maps, settings, fsi, total = load_memmaps(files)
    samplerate = np.floor(np.squeeze(settings[0]["ADCSAMPLERATE"]))
    start_index = int(float(start_s) * samplerate) if start_s is not None else 0
    start_f = get_file_index(fsi, start_index)
    if end_s is not None:
        end_index = int(float(end_s) * samplerate)
        if end_index > total:
            end_index = total
    else:
        end_index = start_index + len(maps[start_f])
    end_f = get_file_index(fsi, end_index)
    if start_f == end_f:
        data = scale_raw_data(maps[start_f][start_index - fsi[start_f]:end_index - fsi[start_f]], settings[start_f])
    else:
        data = scale_raw_data(maps[start_f][start_index - fsi[start_f]:], settings[start_f])
        for i in range(start_f + 1, end_f):
            data = np.concatenate((data, scale_raw_data(maps[i], settings[i])))
        data = np.concatenate((data, scale_raw_data(maps[end_f][:end_index - fsi[end_f]], settings[end_f])))
    return data, samplerate


def load_bin(path, start_s, length_s, samplingfreq):
    """print_trace.py:32-39 / noise-fit.py:89-91 — big-endian (curr_pA, volt_mV) records."""
    columntypes = np.dtype([("curr_pA", ">f8"), ("volt_mV", ">f8")])
    current = np.memmap(path, dtype=columntypes, mode="r")["curr_pA"]
    if start_s is None:
        return np.asarray(current)
    return np.asarray(current[int(start_s * samplingfreq):int((start_s + length_s) * samplingfreq)])


def load_legacy_i2(path, start, end, savegain):
    """legacy/minimal_psd.py:188-193 — (>i2 current, >i2 voltage) records times savegain."""
    columntypes = np.dtype([("current", ">i2"), ("voltage", ">i2")])
    m = np.memmap(path, dtype=columntypes, mode="r")["current"]
    return savegain * m[start:end]


# ------------------------------------------------------------------------------ filter
def filter_data(data, samplerate, cutoff, order, padding=1000):
    """plot-trace.py:313-320 — global-median pad + zero-phase Bessel."""
    Wn = 2.0 * float(cutoff) / float(samplerate)
    b, a = bessel(int(order), Wn, "low")
    padded = np.pad(data, pad_width=padding, mode="median")
    return filtfilt(b, a, padded, padtype=None)[padding:-padding]


def filter_data_edge(data, samplerate, cutoff, poles):
    """legacy/bessel-filter.py:124-131 — edge pad by `poles`, scipy-default filtfilt
    (padtype='odd', padlen=3*ntaps) and `[poles:-poles]`: the result has the length of `data`."""
    Wn = 2.0 * float(cutoff) / float(samplerate)
    b, a = bessel(int(poles), Wn, "low")
    padded = np.pad(data, pad_width=int(poles), mode="edge")
    return filtfilt(b, a, padded, method="pad", padlen=None)[int(poles):-int(poles)]


def lfilter_causal(data, samplerate, cutoff, order, steady=True):
    """Forward-only pass of the same design: scipy.signal.lfilter with the steady-state
    initial condition filtfilt uses (scipy/_signaltools.py:4897-4908)."""
    Wn = 2.0 * float(cutoff) / float(samplerate)
    b, a = bessel(int(order), Wn, "low")
    if steady:
        zi = lfilter_zi(b, a)
        y, _ = lfilter(b, a, data, zi=zi * data[0])
        return y
    return lfilter(b, a, data)


def df2t_lfilter(b, a, x, z):
    """Plain restatement of scipy's compiled `_linear_filter` (direct form II transposed,
    no FMA): y = z0 + b0 x; z[j] = z[j+1] + x b[j+1] - y a[j+1].  Bit-identical to
    scipy.signal.lfilter (SURVEY.md Appendix B.4); slow, for small cases only."""
    n = len(a) - 1
    z = np.array(z, dtype=np.float64).copy()
    y = np.empty(len(x), dtype=np.float64)
    for i in range(len(x)):
        xi = x[i]
        yi = z[0] + b[0] * xi
        for j in range(n - 1):
            z[j] = z[j + 1] + xi * b[j + 1] - yi * a[j + 1]
        z[n - 1] = xi * b[n] - yi * a[n]
        y[i] = yi
    return y, z


# --------------------------------------------------------------------------------- PSD
def psd_length(n, samplerate, psd_length_s=None):
    """plot-trace.py:432-437."""
    if psd_length_s is not None:
        length = 2 ** np.ceil(np.log2(float(psd_length_s) * samplerate))
        if length > n:
            length = n
    else:
        length = np.minimum(2 ** 20, n)
    return length


def welch_psd(x, samplerate, nperseg):
    """plot-trace.py:442 / noise-fit.py:92 — scipy.signal.welch with its defaults."""
    return welch(x, samplerate, nperseg=nperseg)


def welch_explicit(x, fs, nperseg):
    """The formula scipy's welch evaluates (SURVEY.md section 2.2): periodic Hann, hop
    L/2, tail dropped, per-segment mean removal, density scaling, one-sided doubling."""
    L = int(nperseg)
    x = np.asarray(x, dtype=np.float64)
    hop = L - L // 2
    nseg = (len(x) - L // 2) // hop
    w = 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(L) / L)
    acc = np.zeros(L // 2 + 1)
    for s in range(nseg):
        seg = x[s * hop:s * hop + L]
        acc += np.abs(np.fft.rfft(w * (seg - seg.mean()))) ** 2
    P = acc / nseg / (fs * np.sum(w * w))
    if L % 2 == 0:
        P[1:-1] *= 2
    else:
        P[1:] *= 2
    return np.arange(L // 2 + 1) * fs / L, P


def integrate_noise(f, Pxx):
    """plot-trace.py:309-311."""
    df = f[1] - f[0]
    return np.sqrt(np.cumsum(Pxx * df))


def update_psd(filtered, samplerate, psd_length_s=None, normalize=False, cutoff=None):
    """plot-trace.py:418-451 without the plotting."""
    bandwidth = 1.0e6 if cutoff is None else float(cutoff)
    length = psd_length(len(filtered), samplerate, psd_length_s)
    end_index = int(np.floor(len(filtered) / length) * length)
    current = np.average(filtered[:end_index])
    f, Pxx = welch(filtered, samplerate, nperseg=length)
    rms = integrate_noise(f, Pxx)
    if normalize:
        Pxx = Pxx / current ** 2
        Pxx = Pxx * bandwidth
        rms = rms / np.absolute(current)
    return f, Pxx, rms, current


def spectrum_sample(raw, samplerate, psdlength, cutoff):
    """noise-fit.py:92-99."""
    f, Pxx = welch(np.absolute(raw), samplerate, nperseg=psdlength)
    inds = f <= cutoff
    length = np.sum(inds) - 1
    f = f[1:length]
    Pxx = Pxx[1:length].copy()
    current = np.absolute(np.average(raw))
    Pxx *= cutoff / current ** 2
    Pxx *= f
    return f, Pxx, current
