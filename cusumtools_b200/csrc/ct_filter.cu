// C-ABI entry points of stage 1 (dequantise + median pad + zero-phase Bessel; plot-trace.py:272-287, 313-320)
// and the exact median of the masked codes that np.pad(mode='median') needs (plot-trace.py:319).
// The filter passes themselves live in ct_filter_seq.cu.
#include "ct_common.cuh"
#include "cusumtools_b200.h"

namespace {
// ------------------------------ exact median of u16 codes ----------------------------
// Sampled histogram (estimate) + exact window count (verification); the host replays the
// reference's scale_raw_data on the selected code(s) so the pad value is bit-identical
// to np.median(scale_raw_data(raw)) (SURVEY.md H5 / Appendix B.2b).
// The samples of a trace fall on a few hundred codes, i.e. on a dozen L2 lines, and the atomics of one line are serialised
// (1 M samples straight into the global histogram: 93 us).  Each CTA therefore tallies into a shared-memory window of 8192
// codes around its first sample and adds the non-empty bins to the global histogram at the end; codes outside the window
// go to the global histogram directly.  (16 global histograms side by side, summed afterwards, were slower than one:
// the 4 MB of zero-fill and the sum cost more than the contention.)
constexpr int kHistWin = 8192;
__global__ void __launch_bounds__(1024) ct_hist_sampled_kernel(const uint16_t* __restrict__ raw, long long n, long long stride,
                                                               unsigned mask, unsigned* __restrict__ hist) {
    __shared__ unsigned sh[kHistWin];
    __shared__ unsigned sbase;
    for (int i = threadIdx.x; i < kHistWin; i += blockDim.x) sh[i] = 0;
    const long long first = (long long)blockIdx.x * blockDim.x * stride;
    if (threadIdx.x == 0) {
        const unsigned c = first < n ? (raw[first] & mask) : 0u;
        sbase = c > kHistWin / 2 ? c - kHistWin / 2 : 0u;
    }
    __syncthreads();
    const unsigned base = sbase;
    long long i = first + (long long)threadIdx.x * stride;
    const long long step = (long long)gridDim.x * blockDim.x * stride;
    for (; i < n; i += step) {
        const unsigned c = raw[i] & mask, d = c - base;
        if (d < (unsigned)kHistWin) atomicAdd(&sh[d], 1u);
        else atomicAdd(&hist[c], 1u);
    }
    __syncthreads();
    for (int k = threadIdx.x; k < kHistWin; k += blockDim.x) {
        const unsigned v = sh[k];
        if (v) atomicAdd(&hist[base + k], v);       // base + k < 65536 + 4096: bins beyond 65535 stay empty (d < window => c <= 65535)
    }
}

// Rank search in a 65 536-bin histogram on the device: out[0] = first bin whose cumulative count reaches ceil(total / 2)
// (the sampled median), out[1] = its count (the density that gives the estimate's standard error), out[2] = total.
// One CTA of 1024 threads, 64 bins each; replaces a cumsum / searchsorted / gather chain of ten small launches.
template <typename T>
__global__ void __launch_bounds__(1024) ct_hist_rank_kernel(const T* __restrict__ hist, long long* __restrict__ out) {
    __shared__ long long part[1024];
    const int t = threadIdx.x;
    long long s = 0;
#pragma unroll 8
    for (int k = 0; k < 64; ++k) s += (long long)hist[t * 64 + k];
    part[t] = s;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {                 // inclusive scan of the 1024 partial sums
        const long long v = t >= o ? part[t - o] : 0;
        __syncthreads();
        part[t] += v;
        __syncthreads();
    }
    const long long total = part[1023], want = (total + 1) / 2;
    const long long before = t ? part[t - 1] : 0;
    if (total > 0 && before < want && part[t] >= want) {
        long long c = before;
        for (int k = 0; k < 64; ++k) {
            const long long h = (long long)hist[t * 64 + k];
            c += h;
            if (c >= want) { out[0] = t * 64 + k; out[1] = h; out[2] = total; break; }
        }
    }
    if (total == 0 && t == 0) { out[0] = 0; out[1] = 0; out[2] = 0; }
}

constexpr int kWin = 8;
// out[0] = #codes < lo ; out[1+i] = #codes == lo + i*step (step = power of two, lo a multiple of it).
// Eight 8-bit in-register counters in two 32-bit words: with a = 8 (code - lo) / step (negative below the window) the
// increment is 1 << a through PTX shl.b32, which CLAMPS shift amounts >= 32 to "all bits out" (result 0), so codes below
// or above the window add nothing without any compare; the sign bit of a is the "below" count.
// Round 2 (second half): the round-1 form ran 6.5 instructions per code, ALL on the ALU pipe (SHF / LEA.HI / LOP3 / IADD3,
// one warp instruction per two cycles and scheduler): ALU-bound at 0.72 of the DRAM rate (ncu: math_pipe_throttle 1.8 per
// issue).  Now the word is masked and shifted once, a = e * k8 + c and the sign a * 2 >> 32 are IMAD / IMAD.HI (FMA pipe:
// the multipliers are kernel arguments so that ptxas cannot turn them back into shifts), which leaves 3.5 ALU instructions
// per code; and a warp reads 2 KB contiguous per batch instead of four 512-byte pieces 4.8 MB apart
// (scripts/ubench/count_bw.cu: 4.6 -> 5.7 TB/s on 2^30 codes).
static __device__ __forceinline__ unsigned shl_clamp(unsigned v, unsigned amt) {
    unsigned r;
    asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(v), "r"(amt));
    return r;
}
// WIDE = false: only the first four window codes are counted (four 8-bit counters); WIDE: eight 4-bit counters in one register,
// spread into 8-bit counters every 8 codes (the forward pass's tally, ct_filter_seq.cu).
template <bool WIDE>
__global__ void __launch_bounds__(256)
ct_count_window_kernel(const uint16_t* __restrict__ raw, long long n, unsigned mask, unsigned lo,
                       unsigned step, unsigned k8, unsigned two, unsigned long long* __restrict__ out /*[1+kWin]*/) {
    const int sh = __ffs(step) - 1;
    const unsigned nlo8 = 0u - (lo >> sh) * 8u;
    unsigned long long tot[1 + kWin];
#pragma unroll
    for (int i = 0; i <= kWin; ++i) tot[i] = 0;
    // WIDE: eight 4-bit counters in c0 (a = 4 (code - lo) / step), spread into the 8-bit counters of ce / co after the 8
    // codes of every 16-byte load; else four 8-bit counters in c0 (a = 8 (code - lo) / step)
    unsigned below = 0, c0 = 0, ce = 0, co = 0;
    const unsigned ka = WIDE ? k8 >> 1 : k8, nloa = WIDE ? 0u - (lo >> sh) * 4u : nlo8;
    auto tally = [&](unsigned e) {                         // e = (code & mask) >> sh
        const unsigned a = e * ka + nloa;                  // |a| < 2^20
        below = __umulhi(a, two) + below;                  // a >> 31
        c0 += shl_clamp(1u, a);
    };
    auto spread = [&]() {                                  // WIDE, at most 8 tallies since the last call
        ce += c0 & 0x0f0f0f0fu; co += (c0 >> 4) & 0x0f0f0f0fu; c0 = 0;
    };
    auto flush = [&]() {
        tot[0] += below; below = 0;
        if (WIDE) {
            spread();
#pragma unroll
            for (int i = 0; i < 4; ++i) { tot[1 + 2 * i] += (ce >> (8 * i)) & 0xffu; tot[2 + 2 * i] += (co >> (8 * i)) & 0xffu; }
            ce = 0; co = 0;
        } else {
#pragma unroll
            for (int i = 0; i < 4; ++i) tot[1 + i] += (c0 >> (8 * i)) & 0xffu;
            c0 = 0;
        }
    };
    const unsigned m2 = mask | (mask << 16);
    auto tally_word = [&](unsigned w) {
        const unsigned p = (w & m2) >> sh;                 // the low bits of the high code are masked: nothing leaks down
        tally(p & 0xffffu); tally(p >> 16);
    };
    const long long nvec = n / 8;
    const uint4* v = reinterpret_cast<const uint4*>(raw);
    const bool aligned = (reinterpret_cast<uintptr_t>(raw) & 15) == 0;
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long nth = (long long)gridDim.x * blockDim.x;
    if (aligned) {
        // a warp reads 2 KB contiguous per batch (4 x 512 bytes), a CTA 16 KB; CTAs stride over the trace in 16 KB pieces;
        // the next batch is on its way while this one is tallied
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        const long long per_cta = 256 * 4;                 // uint4 per piece
        const long long npieces = nvec / per_cta;
        long long pc = blockIdx.x;
        int rounds = 0;
        uint4 q[4], nq[4];
        bool have = pc < npieces;
        if (have) {
            const uint4* b = v + pc * per_cta + warp * 128 + lane;
#pragma unroll
            for (int u = 0; u < 4; ++u) q[u] = ct_ldg_stream(b + u * 32);
        }
        while (have) {
            const long long pn = pc + gridDim.x;
            const bool more = pn < npieces;
            if (more) {
                const uint4* b = v + pn * per_cta + warp * 128 + lane;
#pragma unroll
                for (int u = 0; u < 4; ++u) nq[u] = ct_ldg_stream(b + u * 32);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                tally_word(q[u].x); tally_word(q[u].y); tally_word(q[u].z); tally_word(q[u].w);
                if (WIDE) spread();
            }
            if (++rounds == 7) { flush(); rounds = 0; }     // 32 tallies per round: an 8-bit counter holds 7 rounds
#pragma unroll
            for (int u = 0; u < 4; ++u) q[u] = nq[u];
            pc = pn;
            have = more;
        }
        flush();
        for (long long i = npieces * per_cta + tid; i < nvec; i += nth) {
            const uint4 qq = ct_ldg_stream(v + i);
            tally_word(qq.x); tally_word(qq.y); tally_word(qq.z); tally_word(qq.w);
            flush();
        }
        for (long long k = nvec * 8 + tid; k < n; k += nth) { tally((unsigned)(raw[k] & mask) >> sh); flush(); }
    } else {
        int since = 0;
        for (long long k = tid; k < n; k += nth) {
            tally((unsigned)(raw[k] & mask) >> sh);
            ++since;
            if (WIDE && (since & 7) == 0) spread();
            if (since == 128) { flush(); since = 0; }
        }
    }
    flush();
#pragma unroll
    for (int i = 0; i < 1 + (WIDE ? kWin : kWin / 2); ++i) {
        unsigned long long sum = tot[i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(CT_FULL, sum, o);
        if (ct_lane() == 0 && sum) atomicAdd(&out[i], sum);
    }
}
// The host side of the exact median (pipeline.median_verify) on the device: the two middle order statistics from the
// window counts, the pad of the filter ends (median - subtracted estimate) and whether the window held them.
__global__ void ct_median_verify_kernel(const unsigned long long* __restrict__ c, int nbins, long long k1, long long k2,
                                        unsigned lo, unsigned step, float sub_code, CtMedianResult* __restrict__ r) {
    if (threadIdx.x) return;
    const unsigned long long below = c[0];
    unsigned long long cum = below;
    unsigned c1 = 0, c2 = 0;
    bool have1 = false, have2 = false;
    for (int i = 0; i < nbins; ++i) {
        cum += c[1 + i];
        if (!have1 && cum >= (unsigned long long)k1 + 1) { c1 = lo + (unsigned)i * step; have1 = true; }
        if (!have2 && cum >= (unsigned long long)k2 + 1) { c2 = lo + (unsigned)i * step; have2 = true; }
    }
    const bool ok = below <= (unsigned long long)k1 && have1 && have2;
    r->code1 = ok ? c1 : 0; r->code2 = ok ? c2 : 0;
    r->pad_x = ok ? 0.5f * ((float)c1 + (float)c2) - sub_code : 0.f;
    r->status = ok ? 0u : ((unsigned long long)k1 < below ? 1u : 2u);
}

}  // namespace

// lane-sequential two-pass implementation (ct_filter_seq.cu)
int ct_filtfilt_seq(const void* in, int in_kind, int64_t n, int64_t pad, float sub, uint16_t mask, float scale,
                    float offset, const CtFilterCoef* coef, int H, int forward_only, float* out, void* workspace,
                    int64_t workspace_bytes, const CtFilterStats* stats, cudaStream_t st);
int ct_filter_forward_seq(const void* in, int in_kind, int64_t n, int64_t pad, float sub, uint16_t mask, float pad_x,
                          const CtFilterCoef* coef, int H, int64_t origin, int part, uint32_t cw_lo, uint32_t cw_step,
                          int64_t cw_begin, int64_t cw_end, uint64_t* counts9, int64_t from_pos, int64_t to_pos,
                          void* workspace, int64_t workspace_bytes, const float* pad_x_dev, cudaStream_t st);
int ct_filter_backward_seq(int64_t n, int64_t pad, float sub, float scale, float offset, const CtFilterCoef* coef, int H,
                           int64_t origin, float* out, const void* workspace, int64_t workspace_bytes,
                           const CtFilterStats* stats, float* summaries, cudaStream_t st);

extern "C" {

int ct_filter_forward_u16(const uint16_t* raw, int64_t n, int64_t pad, float sub_code, uint16_t mask, float pad_x,
                          const CtFilterCoef* coef, int H, int64_t origin, int part, uint32_t window_lo,
                          uint32_t window_step, int64_t count_begin, int64_t count_end, uint64_t* counts9, int64_t from_pos,
                          int64_t to_pos, void* workspace, int64_t workspace_bytes, void* stream) {
    if (!raw || !coef || n <= 0 || pad < 0 || H < 0 || origin < 0) { ct_set_error("filter_forward: bad argument"); return CT_ERR_ARG; }
    return ct_filter_forward_seq(raw, 0, n, pad, sub_code, mask, pad_x, coef, H, origin, part, window_lo, window_step,
                                 count_begin, count_end, counts9, from_pos, to_pos, workspace, workspace_bytes, nullptr,
                                 (cudaStream_t)stream);
}

int ct_filter_forward_ends_u16(const uint16_t* raw, int64_t n, int64_t pad, float sub_code, uint16_t mask,
                               const float* pad_x_dev, const CtFilterCoef* coef, int H, int64_t origin, void* workspace,
                               int64_t workspace_bytes, void* stream) {
    if (!raw || !coef || !pad_x_dev || n <= 0 || pad < 0 || H < 0 || origin < 0) {
        ct_set_error("filter_forward_ends: bad argument"); return CT_ERR_ARG;
    }
    return ct_filter_forward_seq(raw, 0, n, pad, sub_code, mask, 0.f, coef, H, origin, 1, 0, 1, 0, 0, nullptr, 0, 0, workspace,
                                 workspace_bytes, pad_x_dev, (cudaStream_t)stream);
}

int ct_median_verify(const uint64_t* counts9, int nbins, int64_t k1, int64_t k2, uint32_t lo, uint32_t step, float sub_code,
                     CtMedianResult* result, void* stream) {
    if (!counts9 || !result || nbins < 1 || nbins > 8 || k1 < 0 || k2 < k1 || step < 1) {
        ct_set_error("median_verify: bad argument"); return CT_ERR_ARG;
    }
    CT_COUNT_LAUNCH();
    ct_median_verify_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(reinterpret_cast<const unsigned long long*>(counts9), nbins,
                                                                k1, k2, lo, step, sub_code, result);
    return ct_check_launch("ct_median_verify_kernel");
}

int ct_filter_backward(int64_t n, int64_t pad, float sub_code, float scale, float offset, const CtFilterCoef* coef, int H,
                       int64_t origin, float* out, const void* workspace, int64_t workspace_bytes, const CtFilterStats* stats,
                       float* chunk_minmax, void* stream) {
    if (!out || !coef || n <= 0 || pad < 0 || H < 0 || origin < 0) { ct_set_error("filter_backward: bad argument"); return CT_ERR_ARG; }
    return ct_filter_backward_seq(n, pad, sub_code, scale, offset, coef, H, origin, out, workspace, workspace_bytes, stats,
                                  chunk_minmax, (cudaStream_t)stream);
}

int ct_filter_seq_tile(void) { return 64; }

int ct_filtfilt_u16(const uint16_t* raw, int64_t n, int64_t pad, float median_code, uint16_t mask,
                    float alpha, float pad_value, const CtFilterCoef* coef, int H,
                    int forward_only, float* out, void* workspace, int64_t workspace_bytes, const CtFilterStats* stats,
                    void* stream) {
    if (!raw || !out || !coef || n < 0 || pad < 0 || H < 0) { ct_set_error("filter: bad argument"); return CT_ERR_ARG; }
    if (n == 0) return CT_OK;
    return ct_filtfilt_seq(raw, 0, n, pad, median_code, mask, alpha, pad_value, coef, H, forward_only, out, workspace,
                           workspace_bytes, stats, (cudaStream_t)stream);
}

int ct_filtfilt_f32(const float* x, int64_t n, int64_t pad, float pad_value, const CtFilterCoef* coef,
                    int H, int forward_only, float* out, void* workspace, int64_t workspace_bytes,
                    const CtFilterStats* stats, void* stream) {
    if (!x || !out || !coef || n < 0 || pad < 0 || H < 0) { ct_set_error("filter: bad argument"); return CT_ERR_ARG; }
    if (n == 0) return CT_OK;
    return ct_filtfilt_seq(x, 1, n, pad, pad_value, 0xffff, 1.f, pad_value, coef, H, forward_only, out, workspace,
                           workspace_bytes, stats, (cudaStream_t)stream);
}

int ct_hist_sampled_u16(const uint16_t* raw, int64_t n, int64_t stride, uint16_t mask,
                        uint32_t* hist65536, void* stream) {
    if (!raw || !hist65536 || n < 0 || stride < 1) { ct_set_error("hist: bad argument"); return CT_ERR_ARG; }
    if (n == 0) return CT_OK;
    long long ns = (n + stride - 1) / stride;
    int threads = 1024;
    long long blocks = (ns + threads - 1) / threads;
    long long cap = (long long)ct_sm_count();
    if (blocks > cap) blocks = cap;
    CT_COUNT_LAUNCH();
    ct_hist_sampled_kernel<<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(raw, n, stride, mask, hist65536);
    return ct_check_launch("ct_hist_sampled_kernel");
}

static int count_window(const uint16_t* raw, int64_t n, uint16_t mask, uint32_t lo, uint32_t step, uint64_t* counts9,
                        bool wide, void* stream) {
    // a mask bit below step would let the vector path shift the high code's low bits into the low code of a word
    if (!raw || !counts9 || n < 0 || step < 1 || (step & (step - 1)) || (lo & (step - 1)) || (mask & (step - 1))) {
        ct_set_error("count_window: bad argument (step must be a power of two, lo and every masked code multiples of it)");
        return CT_ERR_ARG;
    }
    if (n == 0) return CT_OK;
    long long blocks = (long long)ct_sm_count() * 8;
    long long want = (n / 8 + 255) / 256 + 1;
    if (blocks > want) blocks = want;
    CT_COUNT_LAUNCH();
    if (wide)
        ct_count_window_kernel<true><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
            raw, n, mask, lo, step, 8u, 2u, reinterpret_cast<unsigned long long*>(counts9));
    else
        ct_count_window_kernel<false><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
            raw, n, mask, lo, step, 8u, 2u, reinterpret_cast<unsigned long long*>(counts9));
    return ct_check_launch("ct_count_window_kernel");
}

int ct_hist_rank(const void* hist65536, int is_int64, int64_t* out3, void* stream) {
    if (!hist65536 || !out3) { ct_set_error("hist_rank: null pointer"); return CT_ERR_ARG; }
    CT_COUNT_LAUNCH();
    if (is_int64) ct_hist_rank_kernel<long long><<<1, 1024, 0, (cudaStream_t)stream>>>((const long long*)hist65536, (long long*)out3);
    else ct_hist_rank_kernel<unsigned><<<1, 1024, 0, (cudaStream_t)stream>>>((const unsigned*)hist65536, (long long*)out3);
    return ct_check_launch("ct_hist_rank_kernel");
}

int ct_count_window_u16(const uint16_t* raw, int64_t n, uint16_t mask, uint32_t lo, uint32_t step,
                        uint64_t* counts9, void* stream) {
    return count_window(raw, n, mask, lo, step, counts9, true, stream);
}

int ct_count_window4_u16(const uint16_t* raw, int64_t n, uint16_t mask, uint32_t lo, uint32_t step,
                         uint64_t* counts9, void* stream) {
    return count_window(raw, n, mask, lo, step, counts9, false, stream);
}

}  // extern "C"
