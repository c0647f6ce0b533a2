"""The kernels behind the exact median of the masked ADC codes, each against a plain count of the same operation.

The median sets the constant pad of every filtered trace (np.pad(mode='median')), so it has to be exact.  It comes from
  * ct_count_window_u16 / ct_count_window4_u16: #codes < lo and #codes == lo + i*step for eight (four) codes, in packed
    4-bit and 8-bit register counters; a 16-byte vector path for aligned pointers, a scalar path for the rest;
  * ct_hist_sampled_u16: the strided-sample histogram, tallied in a shared window of 8192 codes per CTA around its
    first sample, with codes outside it added to the global histogram directly;
  * ct_hist_rank: the rank search in that histogram (uint32 counts, or int64 after an all_reduce);
  * ct_radix_hist_f32: one digit pass of the radix select behind filters.float_median (float traces);
  * median.search over the device counters: the sampled estimate, the window moves and the full-histogram fallback.
Every count is compared for exact integer equality with torch.bincount / comparisons on the device or np.bincount on
the host, over the masked codes (raw.view(int16) as int32 & mask); every median with the sorted array's order
statistics or np.median in float64.  Sizes that depend on the grid are computed from the device's SM count."""
import ctypes as C

import numpy as np
import pytest
import torch

from cusumtools_b200 import _lib, filters, median, synth
from cusumtools_b200.design import bessel_lowpass

pytestmark = pytest.mark.gpu
CT_ERR_ARG = -1
PIECE = 8192                        # codes per CTA piece of the vector path (256 threads x 4 uint4)
COUNTERS = [("ct_count_window_u16", 8), ("ct_count_window4_u16", 4)]
# (step, mask): every ADC width the median sees, and a mask with its high bits cleared
STEP_MASKS = [(1, 0xFFFF), (2, 0xFFFE), (4, 0xFFFC), (8, 0xFFF8), (16, 0xFFF0), (4, 0x3FFC)]
INIT9 = [3, 1 << 33, 5, 7, 11, 13, 17, 19, 23]     # counts9 before a call: the kernels add to it (and sentinels at 5..8)


@pytest.fixture(scope="module")
def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def count_blocks(sms):
    """CTAs of the window count once the trace is long enough to fill the grid (8 per SM)."""
    return 8 * sms


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def to_i16(v: torch.Tensor) -> torch.Tensor:
    """Codes 0..65535 (int32 / int64) as the int16 view the kernels read as uint16."""
    return (v - ((v & 0x8000) << 1)).to(torch.int16)


def masked(raw: torch.Tensor, mask: int) -> torch.Tensor:
    return raw.to(torch.int32) & mask                 # int16 -> int32 sign-extends; & mask keeps the code's bits


def ref_window(raw: torch.Tensor, mask: int, lo: int, step: int, nbins: int) -> list[int]:
    """#codes < lo, then #codes == lo + i*step for i < nbins (zeros up to 9 entries), counted on the device."""
    out = [0] * 9
    if raw.numel():
        d = masked(raw, mask) - lo
        idx = torch.where(d < 0, 0, torch.where((d % step == 0) & (d < nbins * step), 1 + d // step, nbins + 1))
        out[:nbins + 1] = torch.bincount(idx.flatten(), minlength=nbins + 2)[:nbins + 1].tolist()
    return out


def run_count(name: str, raw: torch.Tensor, mask: int, lo: int, step: int, init=INIT9, n=None) -> tuple[int, list[int]]:
    """The counts after one call over the first `n` codes of `raw` (all of them by default)."""
    counts = torch.tensor(init, dtype=torch.int64, device=raw.device)
    n = raw.numel() if n is None else n
    rc = getattr(_lib.lib(), name)(raw.data_ptr(), n, mask, lo, step, counts.data_ptr(), _stream())
    return rc, counts.tolist()


def check_count(name: str, nbins: int, raw: torch.Tensor, mask: int, lo: int, step: int, what=""):
    rc, got = run_count(name, raw, mask, lo, step)
    assert rc == 0, _lib.lib().ct_last_error()
    want = [a + b for a, b in zip(INIT9, ref_window(raw, mask, lo, step, nbins))]
    assert got == want, (name, what, raw.numel(), hex(mask), lo, step, got, want)


def window_codes(n: int, lo: int, step: int, mask: int, gen: torch.Generator) -> torch.Tensor:
    """Codes on and around the window (from 2 steps below to 3 above its eight codes, some far away), with random
    bits outside the mask, as int16 on the device."""
    g = torch.randint(-2, 11, (n,), generator=gen, device="cuda", dtype=torch.int32)
    v = (lo + g * step).clamp(0, 65535)
    far = torch.randint(0, 65536, (n,), generator=gen, device="cuda", dtype=torch.int32)
    v = torch.where(torch.rand(n, generator=gen, device="cuda") < 0.1, far, v)
    junk = torch.randint(0, 65536, (n,), generator=gen, device="cuda", dtype=torch.int32) & ~mask & 0xFFFF
    return to_i16((v & mask) | junk)


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


# ------------------------------------------------------------------------------------------------------------------
# A. ct_count_window_u16 / ct_count_window4_u16
# ------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name,nbins", COUNTERS)
def test_count_window_every_offset_and_length(name, nbins, count_blocks):
    """Slices buf[k:k+n] for k = 0..8 elements (only k = 0, 8 take the vector path) at lengths on both sides of one
    piece, of the tail loops (whole uint4 after the pieces, the last n mod 8 codes) and of npieces = k x blocks."""
    B = count_blocks
    lengths = [0, 1, 7, 8, 9, 15, 8191, 8192, 8193, PIECE * 2 + 13, PIECE * 3 + 8 * 5,
               PIECE * (B - 1) + 9, PIECE * B - 8, PIECE * B, PIECE * B + 1, PIECE * (B + 1) + 8 * 37 + 3,
               PIECE * 2 * B, PIECE * 2 * B + 8 * 1023 + 7]
    mask, step, lo = 0xFFFC, 4, 40000
    buf = window_codes(max(lengths) + 8, lo, step, mask, _gen(1))
    for n in lengths:
        for k in range(9):
            if n == 0:                                 # (an empty tensor has no data pointer: n = 0 on a live one)
                assert run_count(name, buf[k:], mask, lo, step, n=0) == (0, INIT9)
                continue
            check_count(name, nbins, buf[k:k + n], mask, lo, step, f"offset {k}")


@pytest.mark.parametrize("name,nbins", COUNTERS)
def test_count_window_many_pieces_per_cta(name, nbins, count_blocks):
    """About 14.5 pieces of 8192 codes per CTA: the vector path flushes its 8-bit counters after 7 rounds and goes on;
    the scalar path flushes after every 128 codes of a thread (~460 per thread here)."""
    n = PIECE * count_blocks * 14 + PIECE * (count_blocks // 2) + 8 * 300 + 5
    for step, mask in [(4, 0xFFFC), (1, 0xFFFF)]:
        lo = 32000
        buf = window_codes(n + 3, lo, step, mask, _gen(2 + step))
        for k in (0, 3):
            check_count(name, nbins, buf[k:k + n], mask, lo, step, f"offset {k}")
        del buf


@pytest.mark.parametrize("name,nbins", COUNTERS)
def test_count_window_saturated_counters(name, nbins, count_blocks):
    """Every code in one window bin, each bin in turn (the top nibble lo + 7 step and, for four codes, lo + 3 step
    included), the code below the window and the first code past it: a thread's 8-bit counter takes 32 codes per round
    of the vector path (224 between flushes), 128 between flushes of the scalar path, and a 4-bit counter 8 between
    spreads.  One round, one 128-code batch or one uint4 more before a flush or spread overflows a counter."""
    n = PIECE * count_blocks * 14 + PIECE * (count_blocks // 2) + 8 * 300 + 5
    mask, step, lo = 0xFFFC, 4, 40000
    junk = torch.randint(0, step, (n + 1,), generator=_gen(9), device="cuda", dtype=torch.int32)
    for i in range(-1, nbins + 1):
        buf = to_i16(junk + (lo + i * step))
        for k in (0, 1):
            raw = buf[k:k + n]
            rc, got = run_count(name, raw, mask, lo, step)
            assert rc == 0
            want = list(INIT9)
            if i < 0:
                want[0] += n
            elif i < nbins:
                want[1 + i] += n
            assert got == want, (name, i, k, got, want)
        del buf
    # the same at a size with one piece per CTA at most
    buf = to_i16(junk[:PIECE * 3 + 8 * 3 + 5] + (lo + (nbins - 1) * step))
    for k in (0, 1):
        check_count(name, nbins, buf[k:], mask, lo, step, "small")


@pytest.mark.parametrize("step,mask", STEP_MASKS)
@pytest.mark.parametrize("name,nbins", COUNTERS)
def test_count_window_edges(name, nbins, step, mask):
    """Codes at lo - step (below), at lo + nbins step (the first one the shift clamp drops), far above and far below;
    lo = 0 (nothing below); a window running past the top code; lo past every code (all below)."""
    top = 0xFFFF & mask
    gen = _gen(step * 131 + mask)
    for lo in (0, step, 20000 // step * step, top - 3 * step, top - step, top, top + step):
        n = 50_003
        targets = torch.tensor([lo - step, lo + nbins * step, lo + (nbins - 1) * step, lo, 0, top, lo + 1000 * step,
                                lo - 1000 * step], dtype=torch.int32, device="cuda")
        targets = targets[(targets >= 0) & (targets <= top)]
        pick = torch.randint(0, targets.numel(), (n,), generator=gen, device="cuda")
        v = targets[pick]
        far = torch.randint(0, 65536, (n,), generator=gen, device="cuda", dtype=torch.int32) & mask
        v = torch.where(torch.rand(n, generator=gen, device="cuda") < 0.2, far, v)
        junk = torch.randint(0, 65536, (n,), generator=gen, device="cuda", dtype=torch.int32) & ~mask & 0xFFFF
        buf = to_i16(v | junk)
        for k in (0, 8, 5):
            check_count(name, nbins, buf[k:], mask, lo, step, f"offset {k}")


@pytest.mark.parametrize("name,nbins", COUNTERS)
def test_count_window_rejects_unrepresentable_windows(name, nbins):
    """A step that is not a power of two, an lo that is not a multiple of step, or a mask that keeps bits below step
    (whose codes are no lo + i*step: the vector path would also shift the high code's low bits into the low code)
    return CT_ERR_ARG and leave counts9 as it was; the same codes with a valid pair are counted."""
    n = PIECE * 4 + 9
    buf = window_codes(n + 1, 40000, 4, 0xFFFF, _gen(17))
    for k in (0, 1):
        raw = buf[k:k + n]
        for step, mask, lo in [(3, 0xFFFF, 39999), (6, 0xFFFC, 39996), (0, 0xFFFF, 40000), (12, 0xFFF0, 40008),
                               (4, 0xFFFC, 40002), (8, 0xFFF8, 40004), (4, 0xFFFF, 40000), (4, 0xFFFE, 40000),
                               (8, 0xFFFC, 40000), (2, 0x3FFF, 4000)]:
            rc, got = run_count(name, raw, mask, lo, step)
            torch.cuda.synchronize()
            assert rc == CT_ERR_ARG and got == INIT9, (name, k, step, hex(mask), lo, rc, got)
        check_count(name, nbins, raw, 0xFFFC, 40000, 4, f"offset {k}")


def test_fused_window_count_rejects_unrepresentable_windows():
    """ct_filter_forward_u16 with counts9: the same requirement (its tally indexes the nibble with 4 (code - lo) / step),
    CT_ERR_ARG and counts9 untouched; the valid pair on the same trace and workspace adds the plain count."""
    L = _lib.lib()
    n, pad = 100_003, 1000
    raw = window_codes(n, 40000, 4, 0xFFFF, _gen(19))
    design = bessel_lowpass(8, 2.0 * 1e5 / synth.FS)
    coef, H = filters.make_coef(design), filters.warmup_samples(design)
    wsb = int(L.ct_filtfilt_workspace_bytes(n, pad, H))
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")

    def fwd(mask, lo, step):
        counts = torch.tensor(INIT9, dtype=torch.int64, device="cuda")
        rc = L.ct_filter_forward_u16(raw.data_ptr(), n, pad, 40000.0, mask, 0.0, C.byref(coef), H, 0, 0, lo, step, 0, n,
                                     counts.data_ptr(), 0, n, ws.data_ptr(), wsb, _stream())
        torch.cuda.synchronize()
        return rc, counts.tolist()

    for mask, lo, step in [(0xFFFF, 40000, 4), (0xFFFE, 40000, 4), (0xFFFC, 40002, 4), (0xFFFF, 40001, 2),
                           (0xFFFE, 40001, 2), (0xFFFF, 40000, 3)]:
        rc, got = fwd(mask, lo, step)
        assert rc == CT_ERR_ARG and got == INIT9, (hex(mask), lo, step, rc, got)
    for mask, lo, step in [(0xFFFC, 39988, 4), (0xFFFE, 39994, 2), (0xFFFF, 39997, 1)]:
        rc, got = fwd(mask, lo, step)
        assert rc == 0, L.ct_last_error()
        assert got == [a + b for a, b in zip(INIT9, ref_window(raw, mask, lo, step, 8))], (hex(mask), lo, step)


# ------------------------------------------------------------------------------------------------------------------
# C. ct_hist_sampled_u16
# ------------------------------------------------------------------------------------------------------------------

def hist_sampled(codes: np.ndarray, stride: int, mask: int, h: torch.Tensor | None = None) -> torch.Tensor:
    raw = torch.from_numpy(codes.view(np.int16)).cuda()
    if h is None:
        h = torch.zeros(65536, dtype=torch.int32, device="cuda")
    _lib.check(_lib.lib().ct_hist_sampled_u16(raw.data_ptr(), raw.numel(), stride, mask, h.data_ptr(), _stream()),
               "ct_hist_sampled_u16")
    return h


def trace_codes(kind: str, n: int, stride: int, rng: np.random.Generator) -> np.ndarray:
    """uint16 codes: `cluster` stays in every CTA's shared window, `uniform` mostly leaves it (global atomics),
    `low` / `high` put each CTA's first sample near code 0 / 65535 (window base clamped / window past the last bin),
    `drift` moves by far more than 8192 codes over the trace (most samples far from their CTA's first one)."""
    first = np.arange(0, n, 1024 * stride)             # CTA b starts at sample b * 1024 * stride
    if kind == "cluster":
        v = rng.normal(30000, 300, n)
    elif kind == "uniform":
        v = rng.integers(0, 65536, n)
    elif kind == "low":
        v = rng.integers(0, 12000, n)
        v[first] = rng.integers(0, 40, first.size)
    elif kind == "high":
        v = rng.integers(52000, 65536, n)
        v[first] = rng.integers(65500, 65536, first.size)
    else:
        v = np.linspace(500, 64000, n) + rng.normal(0, 50, n)
    return np.clip(v, 0, 65535).astype(np.uint16)


@pytest.mark.parametrize("kind", ["cluster", "uniform", "low", "high", "drift"])
@pytest.mark.parametrize("stride", [1, 2, 7, 4099])
def test_hist_sampled_matches_bincount(stride, kind, sms):
    rng = np.random.default_rng(stride * 7 + len(kind))
    sizes = [1, 1024 * stride - 1, 1024 * stride, 1024 * stride + 1]
    if stride < 100:
        sizes += [3 * 1024 * stride + 17, sms * 1024 * stride + 1, 2 * sms * 1024 * stride + 12345]   # threads loop
    else:
        sizes += [5 * stride + 3]                                                      # a handful of samples, one CTA
    for n in sizes:
        codes = trace_codes(kind, n, stride, rng)
        for mask in (0xFFFF, 0xFFFC):
            got = hist_sampled(codes, stride, mask).cpu().numpy().view(np.uint32).astype(np.int64)
            want = np.bincount(codes[::stride] & mask, minlength=65536)
            assert np.array_equal(got, want), (stride, kind, hex(mask), n, np.flatnonzero(got != want)[:8])


def test_hist_sampled_adds_to_the_histogram():
    rng = np.random.default_rng(5)
    a, b = trace_codes("uniform", 700_001, 1, rng), trace_codes("drift", 1_300_007, 3, rng)
    h = hist_sampled(a, 1, 0xFFFF)
    hist_sampled(b, 3, 0xFFFF, h)
    want = np.bincount(a, minlength=65536) + np.bincount(b[::3], minlength=65536)
    assert np.array_equal(h.cpu().numpy().astype(np.int64), want)
    # and a tiny stride-1 histogram: the exact branch of median.estimate for every trace under 2^21 samples
    c = np.array([0, 65535, 65535, 4096, 4097, 8191, 8192], dtype=np.uint16)
    assert np.array_equal(hist_sampled(c, 1, 0xFFFF).cpu().numpy().astype(np.int64), np.bincount(c, minlength=65536))


# ------------------------------------------------------------------------------------------------------------------
# D. ct_hist_rank
# ------------------------------------------------------------------------------------------------------------------

def rank_ref(h: np.ndarray) -> list[int]:
    total = int(h.sum())
    if total == 0:
        return [0, 0, 0]
    idx = int(np.searchsorted(np.cumsum(h), (total + 1) // 2))
    return [idx, int(h[idx]), total]


def rank_dev(h: np.ndarray, int64: bool) -> list[int]:
    t = torch.from_numpy(h.astype(np.int64) if int64 else h.astype(np.uint32).view(np.int32)).cuda()
    out = torch.full((3,), -5, dtype=torch.int64, device="cuda")
    _lib.check(_lib.lib().ct_hist_rank(t.data_ptr(), int(int64), out.data_ptr(), _stream()), "ct_hist_rank")
    return out.tolist()


def rank_cases():
    rng = np.random.default_rng(23)
    z = lambda: np.zeros(65536, dtype=np.int64)          # noqa: E731
    cases = {"empty": z()}
    for b in (0, 12345, 65535):
        h = z(); h[b] = 1; cases[f"one in {b}"] = h
        h = z(); h[b] = 1_000_003; cases[f"all in {b}"] = h
    for a in (63, 65471):                              # the half-total reached exactly at a 64-bin thread boundary
        for ca, cb in ((5, 5), (5, 6), (5, 4), (6, 5)):
            h = z(); h[a], h[a + 1] = ca, cb; cases[f"{a}:{ca}/{cb}"] = h
        h = z(); h[a - 60], h[a], h[a + 1], h[a + 60] = 3, 2, 1, 4; cases[f"{a} padded"] = h
    h = z(); h[0], h[7] = 1, 2; cases["odd total"] = h
    h = z(); h[rng.choice(65536, 20, replace=False)] = rng.integers(1, 50, 20); cases["sparse"] = h
    h = z(); h[[3, 65000]] = [7, 7]; cases["two far bins"] = h
    cases["dense"] = np.bincount(np.clip(rng.normal(33000, 900, 1_000_001), 0, 65535).astype(np.int64), minlength=65536)
    cases["uniform"] = rng.integers(0, 1000, 65536)
    return cases


@pytest.mark.parametrize("int64", [False, True])
def test_hist_rank_matches_cumsum(int64):
    for what, h in rank_cases().items():
        assert rank_dev(h, int64) == rank_ref(h), (what, int64)


def test_hist_rank_large_counts():
    """uint32 counts above 2^31 (the int32 path reads them unsigned) and int64 counts whose sum exceeds 2^32."""
    z = lambda: np.zeros(65536, dtype=np.int64)          # noqa: E731
    h = z(); h[100], h[60000] = 3_000_000_000, 2_999_999_999
    assert rank_dev(h, False) == rank_ref(h) == [100, 3_000_000_000, 5_999_999_999]
    h = z(); h[5], h[64], h[65535] = 4_294_967_295, 1, 4_294_967_295
    assert rank_dev(h, False) == rank_ref(h)
    h = z(); h[1], h[2] = (1 << 31) + 5, (1 << 31) - 3
    assert rank_dev(h, False) == rank_ref(h) == [1, (1 << 31) + 5, (1 << 32) + 2]
    rng = np.random.default_rng(29)
    h = z(); h[rng.choice(65536, 300, replace=False)] = rng.integers(1 << 30, 1 << 34, 300)
    assert h.sum() > 1 << 32 and rank_dev(h, True) == rank_ref(h)
    h = z(); h[64], h[65472] = 1 << 40, (1 << 40) + 1
    assert rank_dev(h, True) == rank_ref(h) == [65472, (1 << 40) + 1, (1 << 41) + 1]


# ------------------------------------------------------------------------------------------------------------------
# E. ct_radix_hist_f32 and filters.float_median
# ------------------------------------------------------------------------------------------------------------------

def fkeys(x: np.ndarray) -> np.ndarray:
    """The order-preserving uint32 keys of float32 values."""
    b = x.view(np.uint32)
    return b ^ np.where(b >> 31, np.uint32(0xFFFFFFFF), np.uint32(0x80000000)).astype(np.uint32)


def special_floats(n: int, rng: np.random.Generator) -> np.ndarray:
    """Normal values with +-0, subnormals, +-inf, the largest finite values and ties in one vector."""
    x = rng.normal(0, 50, n).astype(np.float32)
    sub = np.arange(1, 2001, dtype=np.uint32).view(np.float32)
    parts = [np.float32([0.0, -0.0]).repeat(3000), sub, -sub[::3], np.float32([np.inf, -np.inf]).repeat(50),
             np.float32([3.4e38, -3.4e38, 1.17549435e-38, -1.17549435e-38]).repeat(10), np.float32([1.5]).repeat(40000)]
    sp = np.concatenate(parts)
    at = rng.choice(n, sp.size, replace=False)
    x[at] = sp
    return x


@pytest.mark.parametrize("use_abs", [0, 1])
def test_radix_digit_histograms(use_abs, sms):
    """Each of the four digit passes, under the prefix of several target keys: the 256-bin histogram of the digit of
    the keys that carry the prefix, at a size where every thread of the capped grid loops (16 x SMs x 256 threads)."""
    rng = np.random.default_rng(31 + use_abs)
    n = 16 * sms * 256 * 2 + 777
    x = special_floats(n, rng)
    keys = fkeys(np.abs(x) if use_abs else x)
    srt = np.sort(keys)
    xd = torch.from_numpy(x).cuda()
    targets = {srt[n // 2], srt[0], srt[-1], srt[n // 4], fkeys(np.float32([0.0]))[0], fkeys(np.float32([-0.0]))[0],
               fkeys(np.float32([1.5]))[0], fkeys(np.float32([1e-43]))[0]}
    for t in sorted(targets):
        for p in range(4):
            bits = 8 * p
            prefix = int(t) >> (32 - bits) if bits else 0
            h = torch.zeros(256, dtype=torch.int64, device="cuda")
            _lib.check(_lib.lib().ct_radix_hist_f32(xd.data_ptr(), n, prefix, bits, use_abs, h.data_ptr(), _stream()),
                       "ct_radix_hist_f32")
            sel = keys if not bits else keys[(keys >> np.uint32(32 - bits)) == prefix]
            want = np.bincount((sel >> np.uint32(24 - bits)) & 0xFF, minlength=256)
            assert np.array_equal(h.cpu().numpy(), want), (hex(int(t)), p, use_abs)


def float_median_cases(sms):
    rng = np.random.default_rng(37)
    cap = 16 * sms * 256
    a = np.float32(1.25)
    b = np.nextafter(a, np.float32(np.inf))                  # differs from a in the last digit pass only
    half = cap + 1001
    two = np.concatenate((np.full(half, a), np.full(half, b), rng.normal(0, 1, 2000).astype(np.float32),
                          np.float32([1e6]).repeat(2000)))
    one = np.concatenate((np.full(half + 5, a), np.full(half - 5, b)))
    zeros = np.float32([-0.0, 0.0])
    cases = {
        "n1": np.float32([3.5]), "n2": np.float32([1.0, -2.0]), "n3": np.float32([5.0, -1.0, 2.0]),
        "5M": rng.normal(7, 3, 5_000_000).astype(np.float32),
        "2^24+3": rng.normal(-40, 9, (1 << 24) + 3).astype(np.float32),
        "special": special_floats(cap * 2 + 11, rng),
        "-0/+0 even": zeros.repeat(500), "-0/+0 odd": np.concatenate((zeros.repeat(500), [np.float32(-0.0)])),
        "-0 then +0": np.float32([-0.0] * 3 + [0.0] * 3 + [-1.0, 1.0]),
        "subnormal": np.concatenate((np.arange(1, 4001, dtype=np.uint32).view(np.float32),
                                     -np.arange(1, 3001, dtype=np.uint32).view(np.float32))),
        "inf high": np.float32([np.inf] * 6 + [1.0] * 5), "inf low": np.float32([-np.inf] * 6 + [1.0] * 5),
        "inf even": np.float32([np.inf] * 5 + [2.0] * 5),
        "all equal": np.full(cap + 3, np.float32(-7.75)), "all equal even": np.full(2 * cap, np.float32(0.1)),
        "ties in two values": two, "ties in one value": one,
        "ties at the split": np.float32([1.0] * 7 + [2.0] * 7),
    }
    for k in list(cases):
        cases[k] = rng.permutation(cases[k])
    return cases


def test_float_median_matches_numpy(sms):
    for what, x in float_median_cases(sms).items():
        got = filters.float_median(torch.from_numpy(np.ascontiguousarray(x)).cuda())
        want = float(np.median(x.astype(np.float64)))
        assert got == want, (what, x.size, got, want)


def test_float_median_of_magnitudes(sms):
    rng = np.random.default_rng(41)
    for n in (1, 2, 1_000_000, 16 * sms * 256 * 3 + 1):
        x = rng.normal(0.5, 2, n).astype(np.float32)
        got = filters.float_median(torch.from_numpy(x).cuda(), use_abs=True)
        assert got == float(np.median(np.abs(x).astype(np.float64))), n
    x = special_floats(16 * sms * 256 + 2, rng)
    assert filters.float_median(torch.from_numpy(x).cuda(), use_abs=True) == float(np.median(np.abs(x).astype(np.float64)))


# ------------------------------------------------------------------------------------------------------------------
# F. median.search over the device counters, n > 2^21 (the sampled estimate and the window search run)
# ------------------------------------------------------------------------------------------------------------------

def logged(hist_fn, count_fn, log):
    def h(stride):
        log.append(("hist", int(stride)))
        return hist_fn(stride)

    def c(lo, step):
        log.append(("count", int(lo), int(step)))
        return count_fn(lo, step)
    return h, c


def host_counters(codes: np.ndarray, mask: int):
    """The same search inputs from numpy counts (CPU tensors: median.estimate ranks on the host)."""
    m = codes.astype(np.int64) & mask

    def hist_fn(stride):
        return torch.from_numpy(np.bincount(m[::stride], minlength=65536))

    def count_fn(lo, step):
        d = m - lo
        inside = (d >= 0) & (d < 8 * step) & (d % step == 0)
        return torch.tensor([int((d < 0).sum())] + np.bincount(d[inside] // step, minlength=8).tolist(), dtype=torch.int64)
    return hist_fn, count_fn


def search_both(codes: np.ndarray, mask: int):
    """median.search with the device counters and with host counts: the pair, and the counters each asked for."""
    raw = torch.from_numpy(codes.view(np.int16)).cuda()
    dev_log, host_log = [], []
    got = median.search(raw.numel(), mask, *logged(*median.device_counters(raw, mask), dev_log))
    host = median.search(codes.size, mask, *logged(*host_counters(codes, mask), host_log))
    srt = np.sort(codes.astype(np.int64) & mask)
    want = (int(srt[(codes.size - 1) // 2]), int(srt[codes.size // 2]))
    assert got == want and host == want, (got, host, want)
    assert dev_log == host_log, (dev_log, host_log)
    return dev_log


def periodic(n: int, a: int, b: int) -> np.ndarray:
    """Code a at the sampled positions (i = 0 mod n >> 20), b everywhere else."""
    codes = np.full(n, b, dtype=np.uint16)
    codes[::n >> 20] = a
    return codes


@pytest.mark.parametrize("direction", [1, -1])
def test_search_recovers_from_a_wrong_estimate(direction):
    """The sample sees only a; the median is b, 20 code steps away: the first window misses, the re-estimate gives the
    same window, and 6-step moves reach b within the 16 attempts."""
    n, mask, step = 3 * (1 << 20) + 4097, 0xFFFC, 4
    a = 30000
    log = search_both(periodic(n, a, a + direction * 20 * step), mask)
    hists = [e[1] for e in log if e[0] == "hist"]
    counts = [e for e in log if e[0] == "count"]
    assert hists == [3, 3] and 3 <= len(counts) < 16, log


def test_search_falls_back_to_the_full_histogram():
    """2000 steps between the sampled code and the median: all 16 windows miss, then the full histogram."""
    n, mask = 3 * (1 << 20) + 4097, 0xFFFC
    log = search_both(periodic(n, 20000, 28000), mask)
    assert [e[0] for e in log].count("count") == 16 and log[-1] == ("hist", 1), log


def test_search_on_split_and_extreme_traces():
    rng = np.random.default_rng(43)
    n = (1 << 22) + 2
    lo_c = np.clip(rng.normal(10000, 30, n // 2), 0, 65535)
    hi_c = np.clip(rng.normal(50000, 30, n // 2), 0, 65535)
    split = rng.permutation(np.concatenate((lo_c, hi_c))).astype(np.uint16)   # k1 and k2 in different clusters
    log = search_both(split, 0xFFFC)
    assert log[-1] == ("hist", 1), log
    n = (1 << 21) + 3
    log = search_both(np.full(n, 33332, dtype=np.uint16), 0xFFFC)             # all equal: the first window holds it
    assert [e[0] for e in log] == ["hist", "count"], log
    for mask, top in ((0xFFFC, 65532), (0xFFFF, 65535)):
        for frac0 in (0.55, 0.45):
            n = (1 << 21) + 11
            codes = np.where(rng.random(n) < frac0, 0, top).astype(np.uint16)
            codes |= (rng.integers(0, 65536, n) & ~mask).astype(np.uint16)    # bits the mask drops
            search_both(codes, mask)


def test_four_code_window_verified_on_the_device():
    """The four-code route: median.count_window(nbins=4) at est - step, then median.verify_on_device, against
    median.verify on the same counts and the sorted order statistics; windows above and below the median report
    which way to move."""
    rng = np.random.default_rng(47)
    mask, step = 0xFFFC, 4
    for n in ((1 << 22) + 5, (1 << 22) + 6):
        codes = np.clip(rng.normal(40000, 40, n), 0, 65535).astype(np.uint16) | rng.integers(0, 4, n).astype(np.uint16)
        raw = torch.from_numpy(codes.view(np.int16)).cuda()
        srt = np.sort(codes.astype(np.int64) & mask)
        want = (int(srt[(n - 1) // 2]), int(srt[n // 2]))
        hist_fn, _ = median.device_counters(raw, mask)
        plan = median.estimate(n, mask, hist_fn)
        assert plan.exact is None and plan.se <= 0.25, plan
        for lo, status in ((max(0, plan.est - step), 0), (want[0] + step, 1), (want[1] - 4 * step, 2)):
            plan.lo = lo
            counts = median.count_window(raw, mask, lo, step, torch.zeros(9, dtype=torch.int64, device="cuda"), nbins=4)
            assert counts[5:].tolist() == [0] * 4
            result = torch.zeros(4, dtype=torch.int32, device="cuda")
            median.verify_on_device(plan, counts, 4, result)
            r = result.cpu().numpy()
            pair, new_lo = median.verify(plan, counts)
            assert int(r[3]) == status, (lo, r, want)
            if status == 0:
                assert pair == want and (int(r[0]), int(r[1])) == want
                assert r[2:3].view(np.float32)[0] == np.float32(0.5 * (want[0] + want[1]) - plan.est)
            else:
                assert pair is None and (new_lo < lo) == (status == 1)
