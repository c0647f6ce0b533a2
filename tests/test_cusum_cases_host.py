"""The CUSUM+ path cases of tests/cusum_cases.py mean what they claim, before any kernel runs on them: the C twin (the
reference of the GPU tests) equals the NumPy definition on every window of every case, and the sequential recurrence
on the short windows and the two longest, and every witness holds."""
import numpy as np
import pytest

import cusum_cases as cc
from oracle import events_oracle as eo

NAMES = list(cc.BUILDERS)


@pytest.mark.parametrize("name", NAMES)
def test_witness(name):
    c = cc.BUILDERS[name]()
    assert c.witness and [k for k, v in c.witness.items() if not v] == []


@pytest.mark.parametrize("name", NAMES)
def test_twin_is_the_definition(name):
    c = cc.BUILDERS[name]()
    want = cc.twin(c)
    first, rep = cc.distinct_rows(c)
    for a in want:                                      # a repeated window has the results of its first copy
        assert np.array_equal(a, a[rep])
    sub = cc.subset(c, first)
    x, offs = cc.flat(sub)
    got = eo.cusum_batch(x, offs, c.delta, c.h, c.max_levels)
    for what, a, b in zip(("n_levels", "edges", "mean", "std", "overflow"), got, want):
        assert np.array_equal(a, b[first]), what


@pytest.mark.parametrize("name", NAMES)
def test_twin_is_the_sequential_recurrence(name):
    c = cc.BUILDERS[name]()
    nl, edges, _, _, ovf = cc.twin(c)
    first, _ = cc.distinct_rows(c)
    ok = cc.accepted(c.y, c.w0, c.w1, c.types)[first]
    lens = (c.w1 - c.w0)[first]
    short = first[ok & (lens < 2000)]
    rows = np.concatenate((short[np.linspace(0, short.size - 1, min(short.size, 150)).astype(int)] if short.size else [],
                           first[ok][np.argsort(lens[ok])[-2:]])).astype(int)
    for i in rows:
        ed, o = eo.cusum_event_sequential(c.window(i), c.delta, c.h, c.max_levels)
        assert nl[i] == ed.size - 1 and np.array_equal(edges[i, :ed.size], ed) and ovf[i] == o, i
