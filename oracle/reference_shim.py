"""Headless import of the reference's own scripts (shadowk29/cusumtools, not part of this repository).

The reference is used only when the environment variable CUSUMTOOLS_REFERENCE names a checkout
of it: by tests/golden/make_golden.py (to generate committed fixtures) and by the `not gpu`
tests that re-validate the oracle live against it.  Without it those tests skip and the
committed fixtures pin the oracle.

Recipe from SURVEY.md section 8(c): stub the GUI / dead numpy modules, then load
plot-trace.py and noise-fit.py by path and call the unbound methods of `App` on a
duck-typed `self`.
"""
from __future__ import annotations

import importlib.util
import os
import sys
import types
from types import SimpleNamespace

REFERENCE_ROOT = os.environ.get("CUSUMTOOLS_REFERENCE", "")


def available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isfile(os.path.join(REFERENCE_ROOT, "plot-trace.py"))


def _stub(name: str, **attrs) -> None:
    if name in sys.modules:
        return
    m = types.ModuleType(name)
    for k, v in attrs.items():
        setattr(m, k, v)
    sys.modules[name] = m


_loaded: dict[str, types.ModuleType] = {}


def _install_stubs() -> None:
    for n in ("numpy.random.common", "numpy.random.bounded_integers", "numpy.random.entropy"):
        _stub(n)
    try:
        import matplotlib  # noqa: F401
    except Exception:
        _stub("matplotlib", use=lambda *a, **k: None)
        _stub("matplotlib.figure", Figure=object)
        _stub("matplotlib.backends")
        _stub("matplotlib.backends.backend_tkagg", FigureCanvasTkAgg=object, NavigationToolbar2Tk=object,
              NavigationToolbar2TkAgg=object)
        _stub("matplotlib.pyplot")
        _stub("pylab")
    try:
        import tkinter  # noqa: F401
    except Exception:
        _stub("tkinter", Frame=object, Tk=object)
        _stub("tkinter.filedialog")
        sys.modules["tkinter"].filedialog = sys.modules["tkinter.filedialog"]
    try:
        import pandasql  # noqa: F401
    except Exception:
        _stub("pandasql", sqldf=lambda *a, **k: None)
    if "pylab" not in sys.modules:
        _stub("pylab")


def load(script: str) -> types.ModuleType:
    """Import `$CUSUMTOOLS_REFERENCE/<script>` (e.g. 'plot-trace.py') as a module."""
    if script in _loaded:
        return _loaded[script]
    if not available():
        raise FileNotFoundError(f"reference not found: set CUSUMTOOLS_REFERENCE to a cusumtools checkout "
                                f"(now {REFERENCE_ROOT!r})")
    _install_stubs()
    name = "ref_" + script.replace("-", "_").replace(".py", "").replace(os.sep, "_")
    spec = importlib.util.spec_from_file_location(name, os.path.join(REFERENCE_ROOT, script))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    _loaded[script] = mod
    return mod


class _Entry:
    def __init__(self, v):
        self.v = v

    def get(self):
        return self.v


class _Wild:
    def __init__(self):
        self.msg = None

    def set(self, s):
        self.msg = s


def make_app(samplerate, cutoff=None, order=None, data=None):
    """Duck-typed `self` for the unbound App methods of plot-trace.py."""
    return SimpleNamespace(samplerate=samplerate, wildcard=_Wild(),
                           cutoff_entry=_Entry("" if cutoff is None else str(cutoff)),
                           order_entry=_Entry("" if order is None else str(order)),
                           data=data)


def ref_scale_raw_data(raw_u16, settings, samplerate):
    pt = load("plot-trace.py")
    return pt.App.scale_raw_data(make_app(samplerate), raw_u16, settings)


def ref_filter_data(data, samplerate, cutoff, order):
    pt = load("plot-trace.py")
    app = make_app(samplerate, cutoff, order, data)
    pt.App.filter_data(app)
    return app.filtered_data


def ref_filter_data_edge(data, fc_khz, fs_khz, poles):
    """legacy/bessel-filter.py:124-131 (App.filter_data of the step-response tool): edge pad by `poles`,
    scipy-default filtfilt (odd extension), [poles:-poles].  The tool's entries hold kHz."""
    bf = load(os.path.join("legacy", "bessel-filter.py"))
    app = SimpleNamespace(fc_entry=_Entry(repr(float(fc_khz))), fs_entry=_Entry(repr(float(fs_khz))),
                          poles=_Entry(str(int(poles))), perfect_data=data)
    bf.App.filter_data(app)
    return app.filtered_data


def ref_integrate_noise(f, Pxx):
    pt = load("plot-trace.py")
    return pt.App.integrate_noise(make_app(1.0), f, Pxx)


def ref_load_series(first_file):
    """Run get_filenames + load_memmaps + initialize_samplerate on a .log series."""
    pt = load("plot-trace.py")
    app = make_app(0.0)
    pt.App.get_filenames(app, first_file)
    pt.App.load_memmaps(app)
    pt.App.initialize_samplerate(app)
    app.get_file_index = lambda n: pt.App.get_file_index(app, n)
    app.scale_raw_data = lambda t, s: pt.App.scale_raw_data(app, t, s)
    return pt, app


def ref_load_mapped_data(first_file, start_s, end_s):
    pt, app = ref_load_series(first_file)
    app.start_entry = _Entry("" if start_s is None else repr(float(start_s)))
    app.end_entry = _Entry("" if end_s is None else repr(float(end_s)))
    pt.App.load_mapped_data(app)
    return app.data, app.samplerate


def ref_spectrum_sample(tracefile, samplerate, psdlength, cutoff):
    nf = load("noise-fit.py")
    import contextlib, io
    with contextlib.redirect_stdout(io.StringIO()):
        s = nf.SpectrumSample(tracefile, samplerate, psdlength, cutoff)
    return s
