// Baseline block statistics + threshold/hysteresis event detection with stream compaction.
//
// The reference has no implementation of this stage; the semantics are the consumer's
// (plot-trace.py:379-414: start line = baseline - sign*threshold*stdev, end line =
// baseline - sign*(threshold-hysteresis)*stdev, per baseline block) and the definition is
// oracle/events_oracle.py (block_stats / detect_events).  Everything here is exact:
// block sums are int64 sums of fixed-point samples (order independent), comparisons are
// float32-vs-float32, so event indices are bit-identical to the oracle on the same input.
//
// Detection is a scan over a 2-state automaton (outside/inside) whose per-sample maps are
// "set inside" (A), "set outside" (B) or identity.  Pass 1 reads the trace once
// (4 B/sample), ballots A/B into bit masks (0.25 B/sample written) and emits one summary
// per 4096-sample run; a single-CTA scan chains the run states and prefix-sums the event
// counts; pass 2 reads only the masks and writes start/end indices in time order.
// Inside a 32-sample word the automaton is evaluated with one 64-bit ADD (generate = A,
// propagate = ~(A|B): the carry chain of the adder is the state).
#include "ct_common.cuh"
#include "cusumtools_b200.h"

namespace {

constexpr int kRun = 4096;           // samples per warp run (128 mask words)
constexpr int kRunWords = kRun / 32;
constexpr int kDetWarps = 8;

struct RunSummary {                  // 16 bytes
    unsigned first_last;             // first symbol (bits 0-1), last symbol (bits 2-3); 0 none, 1 in, 2 out
    unsigned ns0;                    // starts assuming the run begins outside
    unsigned ne0;                    // ends   assuming the run begins outside
    unsigned pad;
};

// state after each bit given carry-in c (1 = inside): returns I mask, updates c
__device__ __forceinline__ unsigned automaton_word(unsigned A, unsigned B, unsigned& c) {
    unsigned P = ~(A | B);
    unsigned long long X = (unsigned long long)(A | P), Y = (unsigned long long)A;
    unsigned long long sum = X + Y + c;
    unsigned long long cin = sum ^ X ^ Y;       // bit i = carry into bit i = state before sample i
    unsigned I = (unsigned)(cin >> 1);          // state after sample i
    c = I >> 31;
    return I;
}

// Pass 1: one warp per run of 4096 samples, 1024 samples (32 mask words) per batch.  The 32
// coalesced loads of a batch are independent (deep memory-level parallelism); lane w keeps
// the ballots of row w, so the automaton of all 32 words is evaluated in parallel, one word
// per lane, after a ballot-based resolution of the word-to-word carry (a word is either the
// identity or a constant map on the state).
__global__ void __launch_bounds__(kDetWarps * 32)
ct_detect_pass1(const float* __restrict__ y, long long n, long long block,
                const int* __restrict__ sign, const float* __restrict__ t_start,
                const float* __restrict__ t_end, uint2* __restrict__ masks,
                RunSummary* __restrict__ summ, long long nruns) {
    const int lane = ct_lane();
    const int wib = threadIdx.x >> 5;
    const long long run = (long long)blockIdx.x * kDetWarps + wib;
    if (run >= nruns) return;
    __shared__ uint2 s_ab[kDetWarps][32];        // the 32 ballot pairs of a batch, one row per warp
    const long long base = run * kRun;
    // block is a multiple of kRun, so a run never straddles two baseline blocks
    const long long kb = base / block;
    // a negative baseline mirrors the comparisons: work on sgn*v so that "beyond the start line" is always
    // v' < ts' and "back beyond the end line" always v' > te' (x -> -x is exact, comparisons are unchanged)
    const float sgn = sign[kb] > 0 ? 1.f : -1.f;
    const float ts = sgn * t_start[kb], te = sgn * t_end[kb];
    const bool full = base + kRun <= n;
    unsigned cin = 0, first = 0, last = 0, ns = 0, ne = 0;
    for (int b = 0; b < kRun / 1024; ++b) {
        const long long bb = base + b * 1024;
#pragma unroll
        for (int w0 = 0; w0 < 32; w0 += 8) {
            float v[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const long long p = bb + (w0 + j) * 32 + lane;
                v[j] = (full || p < n) ? sgn * y[p] : te;    // == te is neither symbol
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const unsigned A = __ballot_sync(CT_FULL, v[j] < ts);
                const unsigned B = __ballot_sync(CT_FULL, v[j] > te);
                if (lane == 0) s_ab[wib][w0 + j] = make_uint2(A, B);     // one predicated 64-bit store per row
            }
        }
        __syncwarp();
        const uint2 ab = s_ab[wib][lane];          // lane w owns the ballots of row w
        __syncwarp();
        const unsigned myA = ab.x, myB = ab.y;
        masks[run * kRunWords + b * 32 + lane] = make_uint2(myA, myB);
        const unsigned nz = myA | myB;
        const unsigned lastIn = nz ? ((myA >> (31 - __clz(nz))) & 1u) : 0u;
        const unsigned firstIn = nz ? ((myA >> (__ffs(nz) - 1)) & 1u) : 0u;
        const unsigned nzmask = __ballot_sync(CT_FULL, nz != 0);
        const unsigned lastmask = __ballot_sync(CT_FULL, lastIn != 0);
        const unsigned firstmask = __ballot_sync(CT_FULL, firstIn != 0);
        const unsigned lower = nzmask & ((1u << lane) - 1u);
        unsigned c = lower ? ((lastmask >> (31 - __clz(lower))) & 1u) : cin;
        const unsigned cprev = c;
        const unsigned I = automaton_word(myA, myB, c);
        const unsigned prev = (I << 1) | cprev;
        ns += __popc(I & ~prev);
        ne += __popc(~I & prev);
        if (nzmask) {
            if (!first) first = ((firstmask >> (__ffs(nzmask) - 1)) & 1u) ? 1u : 2u;
            const unsigned hi = 31 - __clz(nzmask);
            cin = (lastmask >> hi) & 1u;
            last = cin ? 1u : 2u;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { ns += __shfl_xor_sync(CT_FULL, ns, o); ne += __shfl_xor_sync(CT_FULL, ne, o); }
    if (lane == 0) {
        RunSummary s; s.first_last = first | (last << 2); s.ns0 = ns; s.ne0 = ne; s.pad = 0;
        summ[run] = s;
    }
}

// Pass 1 from chunk extrema.  The filter's backward pass leaves (min, max) of every 64-sample chunk of its output
// (ct_filter_backward, chunk_minmax); against the block's two lines a chunk is almost always decided as a whole -
// every sample back beyond the end line (baseline), every sample beyond the start line (inside a deep event) or
// neither - and only the chunks that hold a crossing are read from the trace (32 lanes x 2 samples, four ballots).
// Same masks, same run summaries as ct_detect_pass1, at 1/32 of its traffic.  One warp per run of 4096 samples;
// lane l owns chunks 2l, 2l+1 = mask words 4l .. 4l+3.
__global__ void __launch_bounds__(kDetWarps * 32)
ct_detect_pass1_minmax(const float* __restrict__ y, long long n, long long block,
                       const int* __restrict__ sign, const float* __restrict__ t_start,
                       const float* __restrict__ t_end, const float2* __restrict__ mm, long long mm_shift,
                       uint2* __restrict__ masks, RunSummary* __restrict__ summ, long long nruns) {
    const int lane = ct_lane();
    const int wib = threadIdx.x >> 5;
    const long long run = (long long)blockIdx.x * kDetWarps + wib;
    if (run >= nruns) return;
    const long long base = run * kRun;
    const long long kb = base / block;
    const float sgn = sign[kb] > 0 ? 1.f : -1.f;
    const float ts = sgn * t_start[kb], te = sgn * t_end[kb];
    const long long c0 = (base + mm_shift) >> 6;             // first chunk of the run
    unsigned A[4], B[4];
    bool mixed[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const long long cb = base + (2 * lane + k) * 64;     // first sample of the chunk
        bool mix = true;
        unsigned a = 0, b = 0;
        if (cb + 64 <= n) {
            const float2 e = mm[c0 + 2 * lane + k];
            const float lo = sgn > 0.f ? e.x : -e.y, hi = sgn > 0.f ? e.y : -e.x;     // extrema of sgn * v
            if (hi < ts) { a = 0xffffffffu; mix = false; }                // every sample beyond the start line
            else if (lo >= ts && lo > te) { b = 0xffffffffu; mix = false; }   // every sample back beyond the end line
            else if (lo >= ts && hi <= te) mix = false;                   // no symbol at all
        } else if (cb >= n) mix = false;                                  // past the data: no symbol
        A[2 * k] = A[2 * k + 1] = a; B[2 * k] = B[2 * k + 1] = b;
        mixed[k] = mix;
    }
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        unsigned todo = __ballot_sync(CT_FULL, mixed[k]);
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const long long p0 = base + (2 * src + k) * 64 + lane, p1 = p0 + 32;
            const float v0 = p0 < n ? sgn * y[p0] : te, v1 = p1 < n ? sgn * y[p1] : te;   // == te is neither symbol
            const unsigned a0 = __ballot_sync(CT_FULL, v0 < ts), b0 = __ballot_sync(CT_FULL, v0 > te);
            const unsigned a1 = __ballot_sync(CT_FULL, v1 < ts), b1 = __ballot_sync(CT_FULL, v1 > te);
            if (lane == src) { A[2 * k] = a0; B[2 * k] = b0; A[2 * k + 1] = a1; B[2 * k + 1] = b1; }
        }
    }
    uint4* mout = reinterpret_cast<uint4*>(masks + run * kRunWords + 4 * lane);
    mout[0] = make_uint4(A[0], B[0], A[1], B[1]);
    mout[1] = make_uint4(A[2], B[2], A[3], B[3]);
    // the lane's four words as one map on the state: identity, or constant = its last symbol
    unsigned lastIn = 0, firstIn = 0, any = 0;
#pragma unroll
    for (int w = 0; w < 4; ++w) {
        const unsigned nz = A[w] | B[w];
        if (nz) {
            if (!any) firstIn = (A[w] >> (__ffs(nz) - 1)) & 1u;
            lastIn = (A[w] >> (31 - __clz(nz))) & 1u;
            any = 1;
        }
    }
    const unsigned nzmask = __ballot_sync(CT_FULL, any != 0);
    const unsigned lastmask = __ballot_sync(CT_FULL, lastIn != 0);
    const unsigned firstmask = __ballot_sync(CT_FULL, firstIn != 0);
    const unsigned lower = nzmask & ((1u << lane) - 1u);
    unsigned c = lower ? ((lastmask >> (31 - __clz(lower))) & 1u) : 0u;     // a run is evaluated as if it began outside
    unsigned ns = 0, ne = 0;
#pragma unroll
    for (int w = 0; w < 4; ++w) {
        const unsigned cprev = c;
        const unsigned I = automaton_word(A[w], B[w], c);
        const unsigned prev = (I << 1) | cprev;
        ns += __popc(I & ~prev);
        ne += __popc(~I & prev);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { ns += __shfl_xor_sync(CT_FULL, ns, o); ne += __shfl_xor_sync(CT_FULL, ne, o); }
    if (lane == 0) {
        unsigned first = 0, last = 0;
        if (nzmask) {
            first = ((firstmask >> (__ffs(nzmask) - 1)) & 1u) ? 1u : 2u;
            last = ((lastmask >> (31 - __clz(nzmask))) & 1u) ? 1u : 2u;
        }
        RunSummary s; s.first_last = first | (last << 2); s.ns0 = ns; s.ne0 = ne; s.pad = 0;
        summ[run] = s;
    }
}

// ---- hierarchical chained scan over run summaries -----------------------------------
// counts of a summary given the true incoming state (1 = inside)
__device__ __forceinline__ void adjusted(const RunSummary& s, unsigned st, unsigned& a, unsigned& b) {
    const unsigned f = s.first_last & 3;
    a = s.ns0; b = s.ne0;
    if (st == 1) { if (f == 1) a -= 1; else if (f == 2) b += 1; }
}
constexpr int kGroup = 64;
// level 1: one thread per group of 64 runs -> group summary (assuming the group starts outside)
__global__ void ct_detect_scan_groups(const RunSummary* __restrict__ summ, long long nruns,
                                      RunSummary* __restrict__ gsum, long long ngroups) {
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= ngroups) return;
    const long long r0 = g * kGroup, r1 = (r0 + kGroup < nruns) ? r0 + kGroup : nruns;
    unsigned st = 2, first = 0, last = 0, ns = 0, ne = 0;
    for (long long r = r0; r < r1; ++r) {
        const RunSummary s = summ[r];
        unsigned a, b; adjusted(s, st, a, b);
        ns += a; ne += b;
        const unsigned f = s.first_last & 3, l = (s.first_last >> 2) & 3;
        if (!first) first = f;
        if (l) { last = l; st = l; }
    }
    RunSummary o; o.first_last = first | (last << 2); o.ns0 = ns; o.ne0 = ne; o.pad = 0;
    gsum[g] = o;
}
// level 3: one thread per group expands the group's state/offsets to its runs
__global__ void ct_detect_scan_expand(const RunSummary* __restrict__ summ, long long nruns,
                                      const uint4* __restrict__ ginfo, const unsigned long long* __restrict__ goffs,
                                      long long ngroups, uint4* __restrict__ runinfo,
                                      unsigned long long* __restrict__ offs) {
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= ngroups) return;
    const long long r0 = g * kGroup, r1 = (r0 + kGroup < nruns) ? r0 + kGroup : nruns;
    unsigned st = ginfo[g].x ? 1u : 2u;
    unsigned long long ns = goffs[2 * g], ne = goffs[2 * g + 1];
    for (long long r = r0; r < r1; ++r) {
        const RunSummary s = summ[r];
        unsigned a, b; adjusted(s, st, a, b);
        runinfo[r] = make_uint4(st == 1 ? 1u : 0u, 0u, 0u, 0u);
        offs[2 * r] = ns; offs[2 * r + 1] = ne;
        ns += a; ne += b;
        const unsigned l = (s.first_last >> 2) & 3;
        if (l) st = l;
    }
}

// single-CTA chained scan over run summaries -> per-run (state_in, start offset, end offset)
__global__ void __launch_bounds__(1024)
ct_detect_scan(const RunSummary* __restrict__ summ, long long nruns, int state_in,
               uint4* __restrict__ runinfo /* x=state_in, y=unused, (z,w) lo words of offsets */,
               unsigned long long* __restrict__ offs /*[nruns][2]*/,
               unsigned long long* __restrict__ counts /*[2]*/) {
    __shared__ unsigned s_last[1024];
    __shared__ unsigned long long s_ns[1024], s_ne[1024];
    __shared__ unsigned s_statein[1024];
    const int tid = threadIdx.x;
    const long long per = (nruns + 1023) / 1024;
    const long long r0 = tid * per, r1 = (r0 + per < nruns) ? r0 + per : nruns;
    // pass A: thread-local last symbol
    unsigned last = 0;
    for (long long r = r0; r < r1; ++r) { unsigned l = (summ[r].first_last >> 2) & 3; if (l) last = l; }
    s_last[tid] = last;
    __syncthreads();
    if (tid == 0) {   // serial chain over 1024 entries: state entering each thread's range
        unsigned st = state_in ? 1u : 2u;
        for (int i = 0; i < 1024; ++i) { s_statein[i] = st; if (s_last[i]) st = s_last[i]; }
    }
    __syncthreads();
    // pass B: counts with the true incoming state
    unsigned st = s_statein[tid];
    unsigned long long ns = 0, ne = 0;
    for (long long r = r0; r < r1; ++r) {
        RunSummary s = summ[r];
        unsigned f = s.first_last & 3, l = (s.first_last >> 2) & 3;
        unsigned a = s.ns0, b = s.ne0;
        if (st == 1) { if (f == 1) a -= 1; else if (f == 2) b += 1; }
        ns += a; ne += b;
        if (l) st = l;
    }
    s_ns[tid] = ns; s_ne[tid] = ne;
    __syncthreads();
    if (tid == 0) {
        unsigned long long a = 0, b = 0;
        for (int i = 0; i < 1024; ++i) {
            unsigned long long ta = s_ns[i], tb = s_ne[i];
            s_ns[i] = a; s_ne[i] = b; a += ta; b += tb;
        }
        counts[0] = a; counts[1] = b;
    }
    __syncthreads();
    // pass C: write per-run state_in and exclusive offsets
    st = s_statein[tid]; ns = s_ns[tid]; ne = s_ne[tid];
    for (long long r = r0; r < r1; ++r) {
        RunSummary s = summ[r];
        unsigned f = s.first_last & 3, l = (s.first_last >> 2) & 3;
        unsigned a = s.ns0, b = s.ne0;
        if (st == 1) { if (f == 1) a -= 1; else if (f == 2) b += 1; }
        runinfo[r] = make_uint4(st == 1 ? 1u : 0u, 0u, 0u, 0u);
        offs[2 * r] = ns; offs[2 * r + 1] = ne;
        ns += a; ne += b;
        if (l) st = l;
    }
}

// pass 2: one thread per run, masks only
__global__ void __launch_bounds__(128)
ct_detect_pass2(const uint2* __restrict__ masks, const uint4* __restrict__ runinfo,
                const unsigned long long* __restrict__ offs, long long nruns,
                long long* __restrict__ starts, long long* __restrict__ ends, long long cap) {
    const long long run = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (run >= nruns) return;
    unsigned c = runinfo[run].x;
    unsigned long long os = offs[2 * run], oe = offs[2 * run + 1];
    const uint4* m4 = reinterpret_cast<const uint4*>(masks + run * kRunWords);
    const long long base = run * kRun;
    for (int w = 0; w < kRunWords; w += 2) {
        uint4 q = m4[w >> 1];
        unsigned AB[2][2] = {{q.x, q.y}, {q.z, q.w}};
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            unsigned A = AB[j][0], B = AB[j][1];
            if ((A | B) == 0) continue;                 // identity word: state unchanged
            unsigned cprev = c;
            unsigned I = automaton_word(A, B, c);
            unsigned prev = (I << 1) | cprev;
            unsigned S = I & ~prev, E = ~I & prev;
            const long long wb = base + (long long)(w + j) * 32;
            while (S) { int b = __ffs(S) - 1; S &= S - 1; if ((long long)os < cap) starts[os] = wb + b; ++os; }
            while (E) { int b = __ffs(E) - 1; E &= E - 1; if ((long long)oe < cap) ends[oe] = wb + b; ++oe; }
        }
    }
}

// ---------------------------------- block statistics ---------------------------------
// oracle/events_oracle.py::block_stats: a sample counts when its whole aligned 64-sample chunk (the last chunk of
// the trace may be shorter) lies inside [bmin, bmax].  Sixteen lanes own a chunk (a float4 each): the chunk's
// verdict is a 16-lane vote, the sums are exact integers (order independent).
constexpr int kStatChunk = 8192;
__global__ void __launch_bounds__(256)
ct_block_stats_kernel(const float* __restrict__ y, long long n, long long block, long long chunks_per_block,
                      float bmin, float bmax, float c0, float scale,
                      long long* __restrict__ cnt, long long* __restrict__ s1, long long* __restrict__ s2) {
    const long long kb = blockIdx.x / chunks_per_block;
    const long long ch = blockIdx.x % chunks_per_block;
    const long long b0 = kb * block + ch * kStatChunk;
    long long b1 = b0 + kStatChunk;
    const long long bend = (kb + 1) * block < n ? (kb + 1) * block : n;
    if (b1 > bend) b1 = bend;
    const int lane = ct_lane();
    const unsigned half_mask = 0xffffu << (lane & 16);           // the 16 lanes that share a 64-sample chunk
    long long c = 0, a = 0, b = 0;
    const bool aligned = (reinterpret_cast<uintptr_t>(y + b0) & 15) == 0;
    // 8192 samples = 32 rounds of 256 threads x 4 consecutive samples (64-sample chunks: 16 adjacent lanes)
    for (long long wb = b0 + (long long)(threadIdx.x & ~31) * 4; wb < b1; wb += 1024) {      // warp-uniform trip count (full-warp votes)
        const long long p0 = wb + lane * 4;
        float v[4] = {0.f, 0.f, 0.f, 0.f};
        int have = 0;
        if (aligned && p0 + 4 <= b1) {
            const uint4 q = ct_ldg_stream(y + p0);
            v[0] = __uint_as_float(q.x); v[1] = __uint_as_float(q.y); v[2] = __uint_as_float(q.z); v[3] = __uint_as_float(q.w);
            have = 4;
        } else {
#pragma unroll
            for (int e = 0; e < 4; ++e) if (p0 + e < b1) { v[e] = y[p0 + e]; have = e + 1; }
        }
        bool ok = true;
#pragma unroll
        for (int e = 0; e < 4; ++e) if (e < have) ok = ok && v[e] >= bmin && v[e] <= bmax;
        const unsigned votes = __ballot_sync(CT_FULL, ok);
        if ((votes & half_mask) == half_mask) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                if (e < have) {
                    const long long q = (long long)__float2ll_rn(__fmul_rn(__fsub_rn(v[e], c0), scale));
                    c += 1; a += q; b += q * q;
                }
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        c += __shfl_xor_sync(CT_FULL, c, o);
        a += __shfl_xor_sync(CT_FULL, a, o);
        b += __shfl_xor_sync(CT_FULL, b, o);
    }
    if (lane == 0 && c) {
        atomicAdd(reinterpret_cast<unsigned long long*>(cnt + kb), (unsigned long long)c);
        atomicAdd(reinterpret_cast<unsigned long long*>(s1 + kb), (unsigned long long)a);
        atomicAdd(reinterpret_cast<unsigned long long*>(s2 + kb), (unsigned long long)b);
    }
}


// ---------------------------- baseline table + thresholds ----------------------------
// oracle/events_oracle.py::baseline_from_stats + thresholds, evaluated on the device with the
// same individually rounded float64 operations (no FMA contraction), so the thresholds the
// detector compares against never leave the GPU:
//   ma = Sq / cnt ; mean = c0 + ma * 2^-shift ; var = Sqq / cnt - ma * ma ;
//   std = sqrt(max(var, 0)) * 2^-shift ; blocks with cnt < min_count inherit the nearest
//   earlier valid block (the first valid one for leading blocks) ;
//   sign = mean >= 0 ? +1 : -1 ; t_start = (float)(mean - (sign*thr) * std) ;
//   t_end = (float)(mean - (sign*(thr - hyst)) * std)           (plot-trace.py:408-411)
__global__ void __launch_bounds__(1024)
ct_baseline_finalize_kernel(const long long* __restrict__ cnt, const long long* __restrict__ s1,
                            const long long* __restrict__ s2, long long nb, double c0, double inv_sc,
                            long long min_count, double thr, double thr_end, double* __restrict__ mean,
                            double* __restrict__ sd, int* __restrict__ sign, float* __restrict__ t_start,
                            float* __restrict__ t_end, int* __restrict__ status) {
    __shared__ long long s_first;
    __shared__ long long s_warp_last[32], s_warp_first[32];
    for (long long k = threadIdx.x; k < nb; k += blockDim.x) {
        const long long c = cnt[k];
        double m = __longlong_as_double(0x7ff8000000000000LL), s = m;
        if (c >= min_count) {
            const double cd = (double)c;
            const double ma = __ddiv_rn((double)s1[k], cd);
            m = __dadd_rn(c0, __dmul_rn(ma, inv_sc));
            double var = __dsub_rn(__ddiv_rn((double)s2[k], cd), __dmul_rn(ma, ma));
            if (!(var > 0.0)) var = 0.0;
            s = __dmul_rn(__dsqrt_rn(var), inv_sc);
        }
        mean[k] = m; sd[k] = s;
    }
    __syncthreads();
    // Inheritance (a block without enough samples takes the nearest earlier valid block, leading ones the
    // first valid block) as a max-scan of "index of the last valid block": every thread owns a contiguous
    // chunk, the chunks' last/first valid indices are scanned over the CTA, then each chunk is filled.
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    const long long per = (nb + blockDim.x - 1) / blockDim.x;
    const long long lo = (long long)threadIdx.x * per, hi = lo + per < nb ? lo + per : nb;
    const long long kNone = 0x7fffffffffffffffLL;
    long long last = -1, first = kNone;
    for (long long k = lo; k < hi; ++k)
        if (cnt[k] >= min_count) { last = k; if (first == kNone) first = k; }
    long long inc = last, fmin = first;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const long long t = __shfl_up_sync(CT_FULL, inc, d);
        if (lane >= d && t > inc) inc = t;
        const long long u = __shfl_xor_sync(CT_FULL, fmin, d);
        if (u < fmin) fmin = u;
    }
    if (lane == 31) s_warp_last[wid] = inc;
    if (lane == 0) s_warp_first[wid] = fmin;
    __syncthreads();
    long long before = -1;                         // last valid block of the earlier warps
    for (int w = 0; w < wid; ++w) if (s_warp_last[w] > before) before = s_warp_last[w];
    long long prev = __shfl_up_sync(CT_FULL, inc, 1);
    if (lane == 0) prev = -1;
    if (before > prev) prev = before;              // last valid block before this thread's chunk
    if (threadIdx.x == 0) {
        long long f = kNone;
        for (int w = 0; w < nwarp; ++w) if (s_warp_first[w] < f) f = s_warp_first[w];
        s_first = f == kNone ? -1 : f;
        *status = f == kNone ? 1 : 0;
    }
    __syncthreads();
    if (s_first < 0) return;
    {
        long long run = prev >= 0 ? prev : s_first;
        double rm = mean[run], rs = sd[run];       // valid blocks are never overwritten
        for (long long k = lo; k < hi; ++k) {
            if (cnt[k] >= min_count) { rm = mean[k]; rs = sd[k]; }
            else { mean[k] = rm; sd[k] = rs; }
        }
    }
    __syncthreads();
    if (s_first < 0) return;
    for (long long k = threadIdx.x; k < nb; k += blockDim.x) {
        const double m = mean[k], s = sd[k];
        const int sg = m >= 0.0 ? 1 : -1;
        sign[k] = sg;
        t_start[k] = __double2float_rn(__dsub_rn(m, __dmul_rn(sg > 0 ? thr : -thr, s)));
        t_end[k] = __double2float_rn(__dsub_rn(m, __dmul_rn(sg > 0 ? thr_end : -thr_end, s)));
    }
}

// ------------------------------ event windows / type codes ---------------------------
// oracle/events_oracle.py::event_windows on the device, with the event count read from
// device memory (counts2 of ct_detect_f32) so no host round trip separates detection from
// CUSUM+.  Events are [starts[i], ends[i]) for i < min(n_starts, n_ends, capacity); only
// events with pos_lo <= start < pos_hi are kept (time shards: the rank whose owned range
// holds the start owns the event; detection itself runs from the left halo on so that the
// state at the first owned sample is right).  The kept events are the index range
// [i0, i0 + count); outputs are written compacted (index i - i0).  out2 = {count, i0}.
__global__ void ct_event_windows_kernel(const long long* __restrict__ starts, const long long* __restrict__ ends,
                                        const unsigned long long* __restrict__ counts2, long long capacity,
                                        long long n_total, long long pos_lo, long long pos_hi, long long padding,
                                        long long minpoints, long long maxpoints, long long* __restrict__ w0,
                                        long long* __restrict__ w1, int* __restrict__ type, long long* __restrict__ out2) {
    long long ne = (long long)min(counts2[0], counts2[1]);
    if (ne > capacity) ne = capacity;
    // starts are sorted: lower bounds of pos_lo and pos_hi by binary search (every thread, L2 resident)
    auto lower = [&](long long pos) {
        long long a = 0, b = ne;
        while (a < b) { const long long m = (a + b) >> 1; if (starts[m] < pos) a = m + 1; else b = m; }
        return a;
    };
    const long long i0 = lower(pos_lo), i1 = lower(pos_hi);
    const long long t0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    if (t0 == 0) { out2[0] = i1 - i0; out2[1] = i0; }
    for (long long i = i0 + t0; i < i1; i += stride) {
        const long long s = starts[i], e = ends[i];
        const long long a = s - padding, b = e + padding, len = e - s;
        const long long prev_end = i > i0 ? ends[i - 1] : (i0 > 0 ? ends[i0 - 1] : 0);
        const long long next_start = i + 1 < ne ? starts[i + 1] : n_total;
        int t = 0;
        if (a < prev_end || b > next_start || a < 0 || b > n_total) t = 4;
        if (len > maxpoints) t = 3;
        if (len < minpoints) t = 2;
        w0[i - i0] = a; w1[i - i0] = b; type[i - i0] = t;
    }
}


// ---------------------------- intra-event threshold crossings --------------------------
// The consumer draws two more lines inside every event (readevents.py:1363-1366: local_baseline -
// intra_threshold * local_stdev and local_baseline - (intra_threshold - intra_hysteresis) * local_stdev,
// sign-mirrored) and shades the (start, end) pairs of rate.csv's intra_crossing_times_us
// (readevents.py:1340-1343, 1366-1367).  Definition of record: oracle/events_oracle.py::intra_crossings -
// the detector's own two-state automaton run over the event window with those lines (of the baseline
// block that holds the event start), starting outside; a crossing still open at the end of the window
// ends there.  One warp per event: 32 samples per ballot pair, the same adder-carry evaluation.
__global__ void __launch_bounds__(256)
ct_intra_crossings_kernel(const float* __restrict__ y, long long ntot, const long long* __restrict__ w0,
                          const long long* __restrict__ w1, const long long* __restrict__ es, long long nev,
                          const long long* __restrict__ nev_dev, long long block, long long nblocks,
                          const int* __restrict__ sign, const float* __restrict__ ts, const float* __restrict__ te,
                          int K, int* __restrict__ count, int* __restrict__ pairs) {
    if (nev_dev) { const long long d = *nev_dev; nev = d < nev ? d : nev; }
    const int lane = ct_lane();
    const long long gw = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long ev = gw; ev < nev; ev += nw) {
        long long a = w0[ev], b = w1[ev];
        const long long org = a;                       // indices are reported relative to the window start
        if (a < 0) a = 0;
        if (b > ntot) b = ntot;
        long long kb = es[ev] / block;
        if (kb < 0) kb = 0;
        if (kb >= nblocks) kb = nblocks - 1;
        const float sg = sign[kb] > 0 ? 1.f : -1.f;
        const float tst = sg * ts[kb], ten = sg * te[kb];      // mirrored: "beyond" is always "below"
        unsigned c = 0;
        int cnt = 0;
        int* out = pairs + ev * 2 * (long long)K;
        for (long long p = a; p < b; p += 32) {
            const long long i = p + lane;
            const bool valid = i < b;
            const float v = valid ? sg * y[i] : 0.f;
            const unsigned A = __ballot_sync(CT_FULL, valid && v < tst);
            const unsigned B = __ballot_sync(CT_FULL, valid && v > ten);
            const unsigned before = c;
            const unsigned I = automaton_word(A, B, c);
            const unsigned prev = (I << 1) | before;
            unsigned m = (I & ~prev) | (~I & prev);    // starts and ends, alternating in time
            if (lane == 0) {
                while (m) {
                    const int bit = __ffs(m) - 1;
                    m &= m - 1;
                    const int idx = (int)(p - org) + bit;
                    if ((I >> bit) & 1u) { if (cnt < K) out[2 * cnt] = idx; }
                    else { if (cnt < K) out[2 * cnt + 1] = idx; ++cnt; }
                }
            }
        }
        if (lane == 0) {
            if (c) { if (cnt < K) out[2 * cnt + 1] = (int)(b - org); ++cnt; }
            count[ev] = cnt;
        }
    }
}

}  // namespace

extern "C" {

int ct_detect_run(void) { return kRun; }

int64_t ct_detect_workspace_bytes(int64_t n) {
    long long nruns = (n + kRun - 1) / kRun;
    if (nruns < 1) nruns = 1;
    // masks + summaries + runinfo + offsets, each 256-byte aligned
    auto al = [](long long b) { return (b + 255) / 256 * 256; };
    long long ng = (nruns + kGroup - 1) / kGroup;
    return al(nruns * kRunWords * 8) + al(nruns * 16) + al(nruns * 16) + al(nruns * 16) + 3 * al(ng * 16);
}

int ct_block_stats_f32(const float* y, int64_t n, int64_t block, float bmin, float bmax, float c0,
                       int shift, int64_t* cnt, int64_t* s1, int64_t* s2, void* stream) {
    if (!y || !cnt || !s1 || !s2 || n < 0 || block <= 0) { ct_set_error("block_stats: bad argument"); return CT_ERR_ARG; }
    if (block % 64) { ct_set_error("block_stats: the baseline block must be a multiple of 64 samples (the chunk of the in-window rule)"); return CT_ERR_ARG; }
    long long nb = (n + block - 1) / block;
    cudaStream_t st = (cudaStream_t)stream;
    if (nb == 0) return CT_OK;
    cudaMemsetAsync(cnt, 0, nb * 8, st); cudaMemsetAsync(s1, 0, nb * 8, st); cudaMemsetAsync(s2, 0, nb * 8, st);
    long long cpb = (block + kStatChunk - 1) / kStatChunk;
    long long grid = nb * cpb;
    if (grid > 0x7fffffffLL) { ct_set_error("block_stats: trace too long for one launch"); return CT_ERR_UNSUPPORTED; }
    CT_COUNT_LAUNCH();
    ct_block_stats_kernel<<<(unsigned)grid, 256, 0, st>>>(y, n, block, cpb, bmin, bmax, c0, ldexpf(1.f, shift), (long long*)cnt, (long long*)s1, (long long*)s2);
    return ct_check_launch("ct_block_stats_kernel");
}

int ct_detect_f32(const float* y, int64_t n, int64_t block, const int32_t* sign, const float* t_start,
                  const float* t_end, int state_in, const float* chunk_minmax, int64_t minmax_shift, void* workspace,
                  int64_t workspace_bytes, int64_t* starts, int64_t* ends, int64_t capacity, uint64_t* counts2, void* stream) {
    if (!y || !sign || !t_start || !t_end || !workspace || !starts || !ends || !counts2 || n < 0) {
        ct_set_error("detect: bad argument"); return CT_ERR_ARG;
    }
    if (block <= 0 || block % kRun) { ct_set_error("detect: baseline block must be a multiple of %d samples", kRun); return CT_ERR_ARG; }
    if (workspace_bytes < ct_detect_workspace_bytes(n)) { ct_set_error("detect: workspace too small"); return CT_ERR_ARG; }
    cudaStream_t st = (cudaStream_t)stream;
    if (n == 0) { cudaMemsetAsync(counts2, 0, 16, st); return CT_OK; }
    long long nruns = (n + kRun - 1) / kRun;
    auto al = [](long long b) { return (b + 255) / 256 * 256; };
    char* w = (char*)workspace;
    uint2* masks = (uint2*)w;            w += al(nruns * kRunWords * 8);
    RunSummary* summ = (RunSummary*)w;   w += al(nruns * 16);
    uint4* runinfo = (uint4*)w;          w += al(nruns * 16);
    unsigned long long* offs = (unsigned long long*)w;  w += al(nruns * 16);
    const long long ng = (nruns + kGroup - 1) / kGroup;
    RunSummary* gsum = (RunSummary*)w;   w += al(ng * 16);
    uint4* ginfo = (uint4*)w;            w += al(ng * 16);
    unsigned long long* goffs = (unsigned long long*)w;
    long long g1 = (nruns + kDetWarps - 1) / kDetWarps;
    if (chunk_minmax && (minmax_shift < 0 || minmax_shift % 64 || (reinterpret_cast<uintptr_t>(chunk_minmax) & 7))) {
        ct_set_error("detect: chunk extrema need an 8-byte aligned array and a shift that is a multiple of 64"); return CT_ERR_ARG;
    }
    CT_COUNT_LAUNCH();
    if (chunk_minmax)
        ct_detect_pass1_minmax<<<(unsigned)g1, kDetWarps * 32, 0, st>>>(y, n, block, sign, t_start, t_end,
                                                                        reinterpret_cast<const float2*>(chunk_minmax), minmax_shift,
                                                                        masks, summ, nruns);
    else
        ct_detect_pass1<<<(unsigned)g1, kDetWarps * 32, 0, st>>>(y, n, block, sign, t_start, t_end, masks, summ, nruns);
    int rc = ct_check_launch("ct_detect_pass1"); if (rc) return rc;
    CT_COUNT_LAUNCH();
    ct_detect_scan_groups<<<(unsigned)((ng + 127) / 128), 128, 0, st>>>(summ, nruns, gsum, ng);
    rc = ct_check_launch("ct_detect_scan_groups"); if (rc) return rc;
    CT_COUNT_LAUNCH();
    ct_detect_scan<<<1, 1024, 0, st>>>(gsum, ng, state_in, ginfo, goffs, (unsigned long long*)counts2);
    rc = ct_check_launch("ct_detect_scan"); if (rc) return rc;
    CT_COUNT_LAUNCH();
    ct_detect_scan_expand<<<(unsigned)((ng + 127) / 128), 128, 0, st>>>(summ, nruns, ginfo, goffs, ng, runinfo, offs);
    rc = ct_check_launch("ct_detect_scan_expand"); if (rc) return rc;
    CT_COUNT_LAUNCH();
    ct_detect_pass2<<<(unsigned)((nruns + 127) / 128), 128, 0, st>>>(masks, runinfo, offs, nruns, (long long*)starts, (long long*)ends, capacity);
    return ct_check_launch("ct_detect_pass2");
}

int ct_baseline_finalize(const int64_t* cnt, const int64_t* s1, const int64_t* s2, int64_t nb, float c0, int shift,
                         int64_t min_count, double threshold, double hysteresis, double* mean, double* stdev,
                         int32_t* sign, float* t_start, float* t_end, int32_t* status, void* stream) {
    if (!cnt || !s1 || !s2 || !mean || !stdev || !sign || !t_start || !t_end || !status || nb < 0) {
        ct_set_error("baseline_finalize: bad argument"); return CT_ERR_ARG;
    }
    // the end line must lie between the start line and the baseline (NaN thresholds, hysteresis 0, stay allowed)
    if (!(hysteresis >= 0.0)) { ct_set_error("baseline_finalize: hysteresis must be >= 0 (a negative one crosses the lines)"); return CT_ERR_ARG; }
    if (nb == 0) return CT_OK;
    CT_COUNT_LAUNCH();
    ct_baseline_finalize_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(
        (const long long*)cnt, (const long long*)s1, (const long long*)s2, nb, (double)c0, ldexp(1.0, -shift), min_count,
        threshold, threshold - hysteresis, mean, stdev, sign, t_start, t_end, status);
    return ct_check_launch("ct_baseline_finalize_kernel");
}

int ct_event_windows(const int64_t* starts, const int64_t* ends, const uint64_t* counts2, int64_t capacity,
                     int64_t n_total, int64_t pos_lo, int64_t pos_hi, int64_t padding, int64_t minpoints, int64_t maxpoints,
                     int64_t* win_start, int64_t* win_end, int32_t* type, int64_t* out2, void* stream) {
    if (!starts || !ends || !counts2 || !win_start || !win_end || !type || !out2 || capacity < 0) {
        ct_set_error("event_windows: bad argument"); return CT_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    cudaMemsetAsync(out2, 0, 16, st);
    if (capacity == 0) return CT_OK;
    long long grid = (capacity + 255) / 256;
    const long long cap = (long long)ct_sm_count() * 8;
    if (grid > cap) grid = cap;
    CT_COUNT_LAUNCH();
    ct_event_windows_kernel<<<(unsigned)grid, 256, 0, st>>>(
        (const long long*)starts, (const long long*)ends, (const unsigned long long*)counts2, capacity, n_total, pos_lo, pos_hi,
        padding, minpoints, maxpoints, (long long*)win_start, (long long*)win_end, type, (long long*)out2);
    return ct_check_launch("ct_event_windows_kernel");
}

int ct_intra_crossings_f32(const float* y, int64_t n_total, const int64_t* win_start, const int64_t* win_end,
                           const int64_t* ev_start, int64_t n_events, const int64_t* n_events_dev, int64_t block,
                           int64_t n_blocks, const int32_t* sign, const float* t_start, const float* t_end,
                           int32_t max_pairs, int32_t* count, int32_t* pairs, void* stream) {
    if (!y || !win_start || !win_end || !ev_start || !sign || !t_start || !t_end || !count || !pairs || n_events < 0) {
        ct_set_error("intra_crossings: bad argument"); return CT_ERR_ARG;
    }
    if (block <= 0 || n_blocks <= 0 || max_pairs < 1) { ct_set_error("intra_crossings: need block > 0, n_blocks > 0, max_pairs >= 1"); return CT_ERR_ARG; }
    if (n_events == 0) return CT_OK;
    long long grid = (n_events + 7) / 8;
    const long long cap = (long long)ct_sm_count() * 8;
    if (grid > cap) grid = cap;
    CT_COUNT_LAUNCH();
    ct_intra_crossings_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(
        y, n_total, (const long long*)win_start, (const long long*)win_end, (const long long*)ev_start, n_events,
        (const long long*)n_events_dev, block, n_blocks, sign, t_start, t_end, max_pairs, count, pairs);
    return ct_check_launch("ct_intra_crossings_kernel");
}


}  // extern "C"
