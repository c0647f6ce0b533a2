"""The route of the exact median without a GPU: where the window counts come from (the forward pass, their own
kernel, none), where they are verified (one device thread or the host loop) and which window is counted."""
import dataclasses

import pytest

from cusumtools_b200 import median

EST, STEP = 40_000, 4


def _plan(se, step=STEP, exact=None):
    return median.MedianPlan(10_000_001, 5_000_000, 5_000_000, step, step.bit_length() - 1, EST, EST - 3 * step,
                             exact=exact, se=se)


# (plan, route keywords, count, on the device, window lo, window codes)
CASES = {
    "exact": (_plan(float("inf"), exact=(EST, EST)), {}, None, False, EST - 3 * STEP, 8),
    "fixed": (_plan(0.1), {"fixed": True}, None, False, EST - 3 * STEP, 8),
    "streamed": (_plan(0.1), {"streamed": True}, "kernel", False, EST - 3 * STEP, 8),
    "se above 0.8": (_plan(0.81), {}, "kernel", False, EST - 3 * STEP, 8),
    "ride": (_plan(0.5), {}, "ride", True, EST - 3 * STEP, 8),
    "ride at se 0.8": (_plan(0.8), {}, "ride", True, EST - 3 * STEP, 8),
    "8-code kernel": (_plan(0.5), {"fused_count": False}, "kernel", True, EST - 3 * STEP, 8),
    "8-code kernel, step 16": (_plan(0.5, step=16), {}, "kernel", True, EST - 3 * 16, 8),
    "4-code kernel": (_plan(0.25), {"fused_count": False}, "kernel", True, EST - STEP, 4),
    "4-code kernel, step 16": (_plan(0.1, step=16), {}, "kernel", True, EST - 16, 4),
}


@pytest.mark.parametrize("name", CASES)
def test_route(name):
    plan, kw, count, device, lo, nbins = CASES[name]
    before = dataclasses.replace(plan)
    assert median.route(plan, **kw) == (count, device, lo, nbins)
    assert plan == before                                # the caller moves plan.lo
