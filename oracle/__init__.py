"""TEST INFRASTRUCTURE — not product code.

CPU restatement of the reference's raw-trace hot path (shadowk29/cusumtools).  Only
`tests/`, `__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference`
leg may import anything from this package, and only as the checker or the timed CPU
baseline.  The product (`cusumtools_b200/`) never imports it and fails loudly when its
CUDA library is missing.

Pinning status (see DESIGN.md "Oracle"):
  * stages 1 and 4 (dequantise, median pad + Bessel filtfilt, Welch PSD, integrate_noise,
    SpectrumSample) restate reference call sequences whose arithmetic lives in numpy/scipy
    (unpinned third-party: scipy 1.18.1 / numpy 2.3.5 in this image).  The reference ships
    no tests or golden vectors, so the restatement is pinned against OUTPUTS OF THE
    REFERENCE ITSELF: `oracle/reference_shim.py` imports the reference's plot-trace.py and
    noise-fit.py headlessly and `tests/golden/make_golden.py` commits input/output vectors.
  * stages 2 and 3 (threshold detection, CUSUM+) have NO implementation in the reference
    (it only consumes their output).  `oracle/events_oracle.py` is the NumPy definition of
    those stages, committed and documented as the reference for them, per BASELINE.json's
    north_star; parity for them is "unpinned by reference tests" by construction.
"""
