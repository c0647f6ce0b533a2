// Batched per-event CUSUM+ level segmentation, one warp per event.
//
// No reference implementation exists (readevents.py only consumes level_current_pA /
// level_duration_us / blockages_pA / stdev_pA / n_levels, :843-846,1297-1306); the
// definition of record is oracle/events_oracle.py::cusum_event, the two-sided CUSUM of
// SURVEY.md Appendix C with every reduction in exact integer arithmetic, so changepoints
// are bit-identical to the sequential definition whatever the scan order:
//   q_k  = rint((x_k - x_0) * 64)                      (int32)
//   d_k  = q_k - q_anchor ; Sd, Sdd = prefix sums of d, d^2 from the anchor   (exact integers: scan-order independent)
//   m, v = running mean / population variance          (float32 from the exact sums: deviations from the anchor are small)
//   s+-  = rint(1024 * (+-delta/v) (d - m -+ delta/2)) (float32 ops, individually rounded; 1/v correctly rounded)
//   S+-  = prefix sums of s+-, g+- = S+- - running min (warp sum scan + warp min scan)
// A jump is detected at the first k with g+ > H or g- > H; the new level starts after the
// last index at which the winning g was 0; the anchor moves to k and the block is redone
// with the new anchor.  Work per block of 256 samples: lane l holds 8 consecutive samples.
#include "ct_common.cuh"
#include "cusumtools_b200.h"

namespace {

constexpr int kE = 8;                 // samples per lane per block
constexpr int kBlk = 32 * kE;         // 256
constexpr float kQ = 64.0f, kSScale = 1024.0f, kSMax = 2097152.0f;
constexpr int kBig = 0x3fffffff;

struct CusumArgs {
    const float* y; long long ntot;
    const long long* w0; const long long* w1; const int* type; long long nev;
    const long long* nev_dev;          // event count read from device memory (NULL: use nev)
    float delta, h; int max_levels;
    int* n_levels; int* edges; double* mean; double* sd; unsigned char* overflow;
    unsigned long long* counter;       // [0] event fetch counter, [1] pending count, [2] pending fetch counter
    int* pending;                      // events left to the warp-cooperative kernel
    const int* order;                  // hand-out order of the thread-per-event kernel (longest windows first); NULL: index order
};

// fused exclusive scan of an int32 and an int64 lane total (one shuffle round trip per step)
__device__ __forceinline__ void warp_excl_add2(int v, long long w, int lane, int& exv, long long& exw, int& totv,
                                               long long& totw) {
    int iv = v; long long iw = w;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int tv = __shfl_up_sync(CT_FULL, iv, d);
        long long tw = __shfl_up_sync(CT_FULL, iw, d);
        if (lane >= d) { iv += tv; iw += tw; }
    }
    totv = __shfl_sync(CT_FULL, iv, 31); totw = __shfl_sync(CT_FULL, iw, 31);
    exv = iv - v; exw = iw - w;
}
// fused exclusive (sum, running-min) scan for both tests: lane aggregates (s, m) with
// m = min over the lane's local prefix; (l) + (r) = (sl + sr, min(ml, sl + mr)).
__device__ __forceinline__ void warp_excl_summin2(int sp, int mp, int sn, int mn, int lane, int& exsp, int& exmp,
                                                  int& exsn, int& exmn, int& totp, int& bminp, int& totn, int& bminn) {
    int a = sp, b = mp, c = sn, d_ = mn;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int ta = __shfl_up_sync(CT_FULL, a, d), tb = __shfl_up_sync(CT_FULL, b, d);
        int tc = __shfl_up_sync(CT_FULL, c, d), td = __shfl_up_sync(CT_FULL, d_, d);
        if (lane >= d) { b = min(tb, ta + b); a += ta; d_ = min(td, tc + d_); c += tc; }
    }
    totp = __shfl_sync(CT_FULL, a, 31); bminp = __shfl_sync(CT_FULL, b, 31);
    totn = __shfl_sync(CT_FULL, c, 31); bminn = __shfl_sync(CT_FULL, d_, 31);
    exsp = __shfl_up_sync(CT_FULL, a, 1); exmp = __shfl_up_sync(CT_FULL, b, 1);
    exsn = __shfl_up_sync(CT_FULL, c, 1); exmn = __shfl_up_sync(CT_FULL, d_, 1);
    if (lane == 0) { exsp = 0; exmp = kBig; exsn = 0; exmn = kBig; }
}
__device__ __forceinline__ int quantise(float x, float x0) {
    return __float2int_rn(__fmul_rn(__fsub_rn(x, x0), kQ));      // (the conversion saturates at the int32 range)
}
// The increments of both tests from the exact sums of the deviations d = q - q_anchor over [k0, k]
// (oracle/events_oracle.py::cusum_increments, operation for operation, all float32).
struct SeqOut { int sp, sn; };
__device__ __forceinline__ float cusum_mean(long long Sd, float rc) { return __fmul_rn(__ll2float_rn(Sd), rc); }
__device__ __forceinline__ SeqOut cusum_tail(long long Sdd, float m, float rc, float t, float dq, float hq) {
    const float v = __fsub_rn(__fmul_rn(__ll2float_rn(Sdd), rc), __fmul_rn(m, m));
    // branch-free: evaluate with a harmless divisor when the variance carries no information, then mask
    const bool ok = v > 0.f;
    const float r = __fmul_rn(dq, __frcp_rn(ok ? v : 1.f));
    float fa = __fmul_rn(__fmul_rn(r, __fsub_rn(t, hq)), kSScale);
    float fb = __fmul_rn(__fmul_rn(-r, __fadd_rn(t, hq)), kSScale);
    fa = fminf(fmaxf(fa, -kSMax), kSMax);
    fb = fminf(fmaxf(fb, -kSMax), kSMax);
    SeqOut o;
    o.sp = ok ? __float2int_rn(fa) : 0;
    o.sn = ok ? __float2int_rn(fb) : 0;
    return o;
}
// highest index k in [lo, hi] among the lane-held candidates (cand = per-lane best or -1)
__device__ __forceinline__ int warp_max(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(CT_FULL, v, o));
    return v;
}

// One event, one warp (windows longer than the thread-per-event limit, or batches too small
// to fill the GPU with one event per lane).
__device__ void warp_event(const CusumArgs& a, const long long ev, const int lane, const int H, const float dq,
                           const float hq, const bool aligned) {
    {
        int* ed = a.edges + ev * (a.max_levels + 1);
        for (int i = lane; i <= a.max_levels; i += 32) ed[i] = -1;
        const long long p0 = a.w0[ev];
        const long long nn = a.w1[ev] - p0;
        if (nn <= 0 || p0 < 0 || a.w1[ev] > a.ntot || nn > 0x3fffffffLL || (a.type && a.type[ev] != 0)) {
            if (lane == 0) { a.n_levels[ev] = 0; a.overflow[ev] = 0; }
            return;
        }
        const int n = (int)nn;
        const float x0 = a.y[p0];
        __syncwarp();
        if (lane == 0) ed[0] = 0;
        int nedge = 1, overflow = 0;
        int k0 = 0;
        int qa = 0;                         // q at the anchor (x0 itself for the first level)
        long long cSq = 0, cSqq = 0;
        int mp = kBig, mn = kBig;           // running min of S+-, relative to the block start
        int argp = 0, argn = 0;             // last index at which g+- was 0
        const long long abase = p0 & ~7LL;  // 32-byte aligned block grid
        int rs = (int)(abase - p0);         // relative index of the block's first sample (<= 0)
        bool fresh = true;
        int q[kE];
        float xn[kE];                       // prefetched samples of the next block
        int pref_rs = -0x7fffffff;
        auto load_block = [&](int rsb, float (&xv)[kE]) {
            const long long pa = p0 + rsb + lane * kE;
            if (aligned && pa >= 0 && pa + kE <= a.ntot) {
                const uint4* p4 = reinterpret_cast<const uint4*>(a.y + pa);
                uint4 lo = __ldg(p4), hi = __ldg(p4 + 1);
                xv[0] = __uint_as_float(lo.x); xv[1] = __uint_as_float(lo.y); xv[2] = __uint_as_float(lo.z); xv[3] = __uint_as_float(lo.w);
                xv[4] = __uint_as_float(hi.x); xv[5] = __uint_as_float(hi.y); xv[6] = __uint_as_float(hi.z); xv[7] = __uint_as_float(hi.w);
            } else {
#pragma unroll
                for (int e = 0; e < kE; ++e) { long long p = pa + e; xv[e] = (p >= 0 && p < a.ntot) ? a.y[p] : x0; }
            }
        };

        while (rs < n && !overflow) {
            const int r0 = rs + lane * kE;
            if (fresh) {                    // quantise this block's samples, prefetch the next block
                float xv[kE];
                if (pref_rs == rs) {
#pragma unroll
                    for (int e = 0; e < kE; ++e) xv[e] = xn[e];
                } else {
                    load_block(rs, xv);
                }
                if (rs + kBlk < n) { load_block(rs + kBlk, xn); pref_rs = rs + kBlk; }
#pragma unroll
                for (int e = 0; e < kE; ++e) q[e] = quantise(xv[e], x0);
            }
            // ---- exact prefix sums of q, q^2 over [k0, k]
            int pq[kE]; long long pqq[kE];
            {
                int aq = 0; long long aqq = 0;
#pragma unroll
                for (int e = 0; e < kE; ++e) {
                    const int k = r0 + e;
                    const int qv = (k >= k0 && k < n) ? q[e] - qa : 0;       // deviation from the anchor sample
                    aq += qv; aqq += (long long)qv * qv;
                    pq[e] = aq; pqq[e] = aqq;
                }
            }
            int totq, exq; long long totqq, exqq;
            warp_excl_add2(pq[kE - 1], pqq[kE - 1], lane, exq, exqq, totq, totqq);
            // ---- log-likelihood increments (fixed point) and their local prefix sums
            int lp[kE], ln[kE];
            {
                int ap = 0, an = 0;
#pragma unroll
                for (int e = 0; e < kE; ++e) {
                    const int k = r0 + e;
                    int sp = 0, sn = 0;
                    if (k > k0 && k < n) {
                        const int cnt = k - k0 + 1;
                        const float rc = __fdiv_rn(1.0f, (float)cnt);
                        const float m = cusum_mean(cSq + exq + pq[e], rc);
                        const float t = __fsub_rn((float)(q[e] - qa), m);
                        const SeqOut o = cusum_tail(cSqq + exqq + pqq[e], m, rc, t, dq, hq);
                        sp = o.sp; sn = o.sn;
                    }
                    ap += sp; an += sn;
                    lp[e] = ap; ln[e] = an;
                }
            }
            // ---- block-relative S and running minima (positions before the anchor hold S = 0)
            int lmp = kBig, lmn = kBig;
#pragma unroll
            for (int e = 0; e < kE; ++e) { lmp = min(lmp, lp[e]); lmn = min(lmn, ln[e]); }
            int totp, totn, bminp, bminn, exp_, exn_, exmp, exmn;
            warp_excl_summin2(lp[kE - 1], lmp, ln[kE - 1], lmn, lane, exp_, exmp, exn_, exmn, totp, bminp, totn, bminn);
#pragma unroll
            for (int e = 0; e < kE; ++e) { lp[e] += exp_; ln[e] += exn_; }
            exmp = min(exmp, mp); exmn = min(exmn, mn);
            // ---- g = S - running min; first detection; last zero of g
            int firste = kE, zp = -1, zn = -1;
            int gpd[kE], gnd[kE];
            {
                int rp = exmp, rn = exmn;
#pragma unroll
                for (int e = 0; e < kE; ++e) {
                    const int k = r0 + e;
                    rp = min(rp, lp[e]); rn = min(rn, ln[e]);
                    gpd[e] = lp[e] - rp; gnd[e] = ln[e] - rn;
                    const bool valid = k > k0 && k < n;
                    if (valid && firste == kE && (gpd[e] > H || gnd[e] > H)) firste = e;
                }
            }
            const unsigned hit = __ballot_sync(CT_FULL, firste < kE);
            int limit = min(rs + kBlk, n) - 1;      // last index to consider for "last zero"
            int kdet = -1, gp_d = 0, gn_d = 0;
            if (hit) {
                const int ld = __ffs(hit) - 1;
                const int ef = __shfl_sync(CT_FULL, firste, ld);
                kdet = rs + ld * kE + ef;
                int mygp = 0, mygn = 0;
#pragma unroll
                for (int e = 0; e < kE; ++e) if (e == ef) { mygp = gpd[e]; mygn = gnd[e]; }
                gp_d = __shfl_sync(CT_FULL, mygp, ld);
                gn_d = __shfl_sync(CT_FULL, mygn, ld);
                limit = kdet;
            }
#pragma unroll
            for (int e = 0; e < kE; ++e) {
                const int k = r0 + e;
                if (k >= k0 && k <= limit) { if (gpd[e] == 0) zp = k; if (gnd[e] == 0) zn = k; }
            }
            zp = warp_max(zp); zn = warp_max(zn);
            if (zp >= 0) argp = zp;
            if (zn >= 0) argn = zn;
            if (hit) {
                const int jmin = (gp_d >= gn_d) ? argp : argn;
                if (nedge >= a.max_levels) { overflow = 1; break; }
                if (lane == 0) ed[nedge] = jmin + 1;
                ++nedge;
                k0 = kdet; cSq = 0; cSqq = 0; mp = kBig; mn = kBig; argp = kdet; argn = kdet;
                qa = quantise(a.y[p0 + kdet], x0);
                // restart at the lane chunk (32-byte grid) that holds the new anchor: nothing before
                // it is needed again, so no block position is spent on samples behind the anchor
                const int nrs = rs + ((kdet - rs) & ~(kE - 1));
                fresh = nrs != rs;                  // same chunk: redo this block with the new anchor
                rs = nrs;
            } else {
                cSq += totq; cSqq += totqq;
                const long long nmp = (long long)min(mp, bminp) - totp, nmn = (long long)min(mn, bminn) - totn;
                mp = (int)max(min(nmp, (long long)kBig), -(long long)kBig);
                mn = (int)max(min(nmn, (long long)kBig), -(long long)kBig);
                rs += kBlk;
                fresh = true;
            }
        }
        if (lane == 0) { ed[nedge] = n; a.n_levels[ev] = nedge; a.overflow[ev] = (unsigned char)overflow; }
        __syncwarp();
        // ---- level statistics from exact integer sums (second, cheap pass; L1/L2 resident)
        for (int i = 0; i < nedge; ++i) {
            const int e0 = ed[i], e1 = ed[i + 1];
            long long sq = 0, sqq = 0;
            for (int k = e0 + lane; k < e1; k += 32) {
                const long long qv = quantise(a.y[p0 + k], x0);
                sq += qv; sqq += qv * qv;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { sq += __shfl_xor_sync(CT_FULL, sq, o); sqq += __shfl_xor_sync(CT_FULL, sqq, o); }
            if (lane == 0) {
                const double len = (double)(e1 - e0), ad = (double)sq, bd = (double)sqq;
                a.mean[ev * a.max_levels + i] = __dadd_rn((double)x0, __ddiv_rn(__ddiv_rn(ad, len), 64.0));
                double var = __dsub_rn(bd, __ddiv_rn(__dmul_rn(ad, ad), len));
                if (var < 0.0) var = 0.0;
                a.sd[ev * a.max_levels + i] = __ddiv_rn(__dsqrt_rn(__ddiv_rn(var, len)), 64.0);
            }
        }
        __syncwarp();
    }
}

// Events the thread-per-event kernel left to the warps (a.pending[0 .. counter[1])): persistent
// warps pull them from an atomic counter, one event per warp at a time.
__global__ void __launch_bounds__(128, 4) ct_cusum_warp_kernel(CusumArgs a) {
    const int lane = ct_lane();
    const int H = __float2int_rn(__fmul_rn(a.h, kSScale));
    const float dq = __fmul_rn(a.delta, kQ);
    const float hq = __fmul_rn(dq, 0.5f);
    const bool aligned = (reinterpret_cast<uintptr_t>(a.y) & 31) == 0;
    const unsigned long long npend = a.counter[1];
    for (;;) {
        unsigned long long i = 0;
        if (lane == 0) i = atomicAdd(a.counter + 2, 1ULL);
        i = __shfl_sync(CT_FULL, i, 0);
        if (i >= npend) break;
        warp_event(a, (long long)a.pending[i], lane, H, dq, hq, aligned);
        __syncwarp();
    }
}

// =====================================================================================
// Thread-per-event kernel (the production path for windows up to kSeqMax samples).
//
// The definition (oracle/events_oracle.py::cusum_event_sequential) is a per-sample recurrence; evaluating it
// literally, one event per LANE, needs no prefix scans, no validity masks, no block re-runs after a detection and
// no second pass for the level statistics.  What decides the speed is how the 32 private sample streams of a warp
// reach the lanes and how many instructions the plateaus of an event cost:
//  * every lane's window is cut into PIECES of 32 samples on the 128-byte line grid of the trace.  A warp moves the
//    next piece of all its 32 lanes with 8 cp.async instructions (8 lanes x 16 bytes = one whole line per event,
//    global -> shared memory without registers, one round ahead), into rows of 144 bytes (bank-conflict-free 128-bit
//    reads of a lane's own row); the 16 spare bytes of a row carry the piece's header (event, index of its first
//    sample, window length, line), written by the fetch cursor of the lane, which runs one round ahead of the
//    evaluation and takes the next event from the shared counter (warp aggregated) when its window is used up;
//  * the reciprocal table of the sample count (1.0f / cnt, IEEE) lives in shared memory, built by the CTA;
//  * the warp is convergent throughout: votes are over all 32 lanes, lanes without a sample at a position vote "yes"
//    and commit nothing.
// Level sums are exact integers: the sums of the samples between the changepoint and the detection index are
// re-read at the (rare) detections, and the float64 mean / std are produced by ct_cusum_finalize from the integer
// sums the lanes leave (bit-cast) in the mean / std arrays.
// =====================================================================================
constexpr int kS = 8;                  // samples a lane processes per (unrolled) group
constexpr int kPiece = 32;             // samples per piece = one 128-byte line
constexpr int kRowB = 144;             // bytes per shared-memory row: 128 of samples + 16 of header
constexpr int kStageB = 32 * kRowB;    // one round of a warp
constexpr int kStages = 2;
#ifndef CT_CUSUM_SEQ_WARPS
#define CT_CUSUM_SEQ_WARPS 20
#endif
constexpr int kSeqWarps = CT_CUSUM_SEQ_WARPS;   // warps per CTA, one CTA per SM
constexpr int kSeqMax = 16384;         // longest window a single lane takes
constexpr int kSeqTab = 8192 + 16;     // entries of the reciprocal table in shared memory
constexpr int kSeqTabLead = 8;         // zero entries in front of it (the positions of a group before the window's first sample)
constexpr int kSeqSmem = (kSeqTab + kSeqTabLead) * 4 + kSeqWarps * kStages * kStageB;
constexpr int kSeqMinEvents = 16384;   // below this one event per lane cannot fill the GPU: warps take everything
constexpr unsigned char kRawSums = 0x80;   // overflow[] bit: level rows hold raw integer sums (finalize pending)

// sums of q, q^2 (relative to x0: what the level statistics are made of) over the cnt samples from the anchor, from
// the sums of the deviations d = q - qa
__device__ __forceinline__ void level_sums(long long Sd, long long Sdd, int cnt, int qa, long long& Sq, long long& Sqq) {
    Sq = Sd + (long long)cnt * qa;
    Sqq = Sdd + 2LL * qa * Sd + (long long)cnt * ((long long)qa * qa);
}
__device__ __forceinline__ void cp_async16(unsigned dst, const void* src, int bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" :: "r"(dst), "l"(src), "r"(bytes) : "memory");
}

__global__ void __launch_bounds__(kSeqWarps * 32, 1) ct_cusum_seq_kernel(CusumArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    float* rct = reinterpret_cast<float*>(smem) + kSeqTabLead;           // rct[-kSeqTabLead .. 0] = 0, rct[c] = 1.0f / c
    const int lane = ct_lane();
    unsigned char* wbuf = smem + (kSeqTab + kSeqTabLead) * 4 + (threadIdx.x >> 5) * (kStages * kStageB);
    for (int i = (int)threadIdx.x - kSeqTabLead; i < kSeqTab; i += blockDim.x) rct[i] = i > 0 ? __fdiv_rn(1.0f, (float)i) : 0.f;
    __syncthreads();
    const int H = __float2int_rn(__fmul_rn(a.h, kSScale));
    const float dq = __fmul_rn(a.delta, kQ);
    const float hq = __fmul_rn(dq, 0.5f);
    long long nev = a.nev;
    if (a.nev_dev) { const long long d = *a.nev_dev; nev = d < nev ? d : nev; }
    const int ML = a.max_levels;
    const bool aligned = (reinterpret_cast<uintptr_t>(a.y) & 15) == 0;      // cp.async moves 16-byte units
    const long long seq_limit = (nev < kSeqMinEvents || !aligned) ? 0 : kSeqMax;
    const long long full_lines = a.ntot >> 5;

    // ---- fetch cursor (one round ahead of the evaluation)
    bool exhausted = false;
    int f_ev = 0, f_n = 0, f_kb = 0, f_left = 0;
    unsigned f_line = 0;
    auto fetch = [&](int stage) {
        unsigned need = __ballot_sync(CT_FULL, f_left == 0 && !exhausted);
        while (need) {                                       // lanes whose window is used up take the next events
            const int leader = __ffs(need) - 1;
            long long base = 0;
            if (lane == leader) base = (long long)atomicAdd(a.counter, (unsigned long long)__popc(need));
            base = __shfl_sync(CT_FULL, base, leader);
            if (f_left == 0 && !exhausted) {
                const long long slot = base + __popc(need & ((1u << lane) - 1u));
                if (slot >= nev) exhausted = true;
                else {
                    const long long ev = a.order ? a.order[slot] : slot;
                    const long long p0 = a.w0[ev];
                    const long long nn = a.w1[ev] - p0;
                    const bool bad = nn <= 0 || p0 < 0 || a.w1[ev] > a.ntot || nn > 0x3fffffffLL || (a.type && a.type[ev] != 0);
                    if (bad) { a.n_levels[ev] = 0; a.overflow[ev] = 0; }
                    else if (nn > seq_limit) a.pending[atomicAdd(a.counter + 1, 1ULL)] = (int)ev;
                    else {
                        f_ev = (int)ev; f_n = (int)nn;
                        f_kb = -(int)(p0 & (kPiece - 1));
                        f_line = (unsigned)(p0 >> 5);
                        f_left = (f_n - f_kb + kPiece - 1) >> 5;
                        a.edges[ev * (ML + 1)] = 0;
                    }
                }
            }
            need = __ballot_sync(CT_FULL, f_left == 0 && !exhausted);
        }
        unsigned char* st = wbuf + stage * kStageB;
        const bool has = f_left > 0;
        *reinterpret_cast<int4*>(st + lane * kRowB + 128) = make_int4(has ? f_ev : -1, f_kb, f_n, (int)f_line);
        // valid samples of the lane's line (32 except on the trace's last line; 0 without a piece: nothing is read)
        int avail = 0;
        if (has) avail = (long long)f_line < full_lines ? kPiece : (int)(a.ntot - ((long long)f_line << 5));
        const unsigned myline = has ? f_line : 0u;
        const unsigned dst0 = (unsigned)__cvta_generic_to_shared(st) + (lane >> 3) * kRowB + (lane & 7) * 16;
        const char* src0 = reinterpret_cast<const char*>(a.y) + (lane & 7) * 16;
        const int c4 = (lane & 7) * 4;
        if (__all_sync(CT_FULL, avail == kPiece)) {          // the usual round: 32 whole lines
#pragma unroll
            for (int it = 0; it < 8; ++it) {                 // 4 rows per instruction, one 128-byte line each
                const unsigned L = __shfl_sync(CT_FULL, myline, it * 4 + (lane >> 3));
                cp_async16(dst0 + it * 4 * kRowB, src0 + ((unsigned long long)L << 7), 16);
            }
        } else {
#pragma unroll
            for (int it = 0; it < 8; ++it) {
                const unsigned L = __shfl_sync(CT_FULL, myline, it * 4 + (lane >> 3));
                const int A = __shfl_sync(CT_FULL, avail, it * 4 + (lane >> 3));
                cp_async16(dst0 + it * 4 * kRowB, src0 + ((unsigned long long)L << 7), min(max(A - c4, 0), 4) * 4);
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        if (has) { ++f_line; f_kb += kPiece; --f_left; }
    };

    // ---- per-lane event state
    bool running = false;                // inside an event that has not been closed
    long long p0 = 0;
    int ev = 0, n = 0;
    float x0 = 0.f, nx0 = 0.f;           // the window's first sample and -64 x0 (quantisation: (x - x0) * 64, one FFMA)
    int k0 = 0, qa = 0, gp = 0, gn = 0, rp = 0, rn = 0, nedge = 1, e0 = 0;
    long long Sd = 0, Sdd = 0;           // sums of d = q - qa, d^2 over [k0, k] (qa = q at the anchor k0)
    long long Lp = 0, Lpp = 0;           // sums of q, q^2 over [e0, k0): the part of the open level before the anchor
    long long ZpS = 0, ZpSS = 0, ZnS = 0, ZnSS = 0;   // sums of d, d^2 over [k0, last zero of g+ / g-] (valid while that g > 0)

#pragma unroll
    for (int s = 0; s < kStages; ++s) fetch(s);
    int stage = 0;
    for (;;) {
        asm volatile("cp.async.wait_group %0;" :: "n"(kStages - 1) : "memory");
        __syncwarp();
        const float* row = reinterpret_cast<const float*>(wbuf + stage * kStageB + lane * kRowB);
        const int4 hdr = *reinterpret_cast<const int4*>(row + kPiece);
        const bool hev = hdr.x >= 0;
        if (__ballot_sync(CT_FULL, hev) == 0) break;         // the cursors ran dry: every later round is empty as well
        const int kb = hdr.y;                                 // window index of the piece's first sample
        if (hev && kb <= 0) {                                 // first piece of the lane's next event
            ev = hdr.x; n = hdr.z;
            p0 = ((long long)(unsigned)hdr.w << 5) - kb;
            x0 = row[-kb];
            nx0 = __fmul_rn(x0, -kQ);
            k0 = 0; qa = 0; gp = gn = 0; rp = rn = 0; nedge = 1; e0 = 0;
            Sd = Sdd = 0; Lp = Lpp = 0;
            running = true;
        }
#pragma unroll 1
        for (int g = 0; g < kPiece / kS; ++g) {
            const int gk = kb + g * kS;
            const bool act = hev && running && gk < n && gk + kS > 0;
            if (!__any_sync(CT_FULL, act)) continue;
            float xv[kS];
            {
                const float4 u = *reinterpret_cast<const float4*>(row + g * kS);
                const float4 v = *reinterpret_cast<const float4*>(row + g * kS + 4);
                xv[0] = u.x; xv[1] = u.y; xv[2] = u.z; xv[3] = u.w; xv[4] = v.x; xv[5] = v.y; xv[6] = v.z; xv[7] = v.w;
            }
            unsigned nlim = act ? (unsigned)n : 0u;
            // ---- quiet prefix.  A sample is QUIET when both statistics are 0 and its deviation from the running mean
            // is within +-delta/2: both increments are then <= 0 whatever the variance is (r > 0 or masked; t - hq <= 0
            // and t + hq >= 0 survive every rounding and the clamps), so the statistics stay 0 with their argmin at the
            // sample - exactly what the full evaluation would leave; only the running sums move.  On the plateaus of an
            // event almost every sample is quiet.  All lanes evaluate the group as if it were quiet (straight-line
            // code on 32-bit sums); the first position at which that is not known to hold for a lane (statistics not 0:
            // position 0; a deviation outside the band: there) goes through one warp reduction, which gives the prefix
            // every lane may commit; the per-sample path takes the rest.  The positions of a group that lie outside the
            // lane's window do not break the prefix: before the window they hold the first sample (deviation 0, the
            // table's zero entries make the mean 0), behind it they are masked and left out of the sums.
            if (__any_sync(CT_FULL, act && gk < 0)) {
#pragma unroll
                for (int e = 0; e < kS - 1; ++e)
                    if (gk + e < 0) xv[e] = x0;
            }
            const int endc = n - gk;                                     // positions of the group inside the window (>= kS: all)
            int dv[kS];
            int s32 = (int)Sd;                                           // (the attempt needs the sum to fit: 32-bit adds and conversions)
            unsigned nq = 0;
            {
                // (counts beyond the shared-memory table - a plateau of more than 8 192 samples - and sums beyond 2^30
                // take the per-sample path)
                const bool att = act && (gp | gn) == 0 && gk - k0 + kS < kSeqTab &&
                                 (unsigned long long)(Sd + (1LL << 30)) < (1ULL << 31);
                const float* rcp = rct + (att ? gk - k0 + 1 : 1);
#pragma unroll
                for (int e = 0; e < kS; ++e) {
                    dv[e] = __float2int_rn(__fmaf_rn(xv[e], kQ, nx0)) - qa;
                    s32 += dv[e];                                        // |d| < 2^23 (the definition's domain): no overflow
                    const float t = __fsub_rn((float)dv[e], __fmul_rn(__int2float_rn(s32), rcp[e]));
                    if (!(fabsf(t) <= hq)) nq |= 1u << e;
                }
                if (endc < kS) nq &= (1u << endc) - 1u;
                nq |= 1u << kS;
                if (!att) nq = 1u;
                if (!act) nq = 1u << kS;
            }
            const int F = (int)__reduce_min_sync(CT_FULL, (unsigned)(__ffs(nq) - 1));
            if (F > 0 && act) {
                if (F == kS && endc >= kS) {
                    Sd = s32;
#pragma unroll
                    for (int e = 0; e < kS; ++e) Sdd += (long long)dv[e] * dv[e];
                } else {
                    const int lim = min(F, endc);
#pragma unroll
                    for (int e = 0; e < kS; ++e)
                        if (e < lim) { Sd += dv[e]; Sdd += (long long)dv[e] * dv[e]; }
                }
                rp = rn = max(gk + F - 1, 0);
            }
            if (F < kS) {
                // (rolled: the evaluation and the changepoint bookkeeping exist once, the code stays in the instruction cache)
#pragma unroll 1
            for (int e = F; e < kS; ++e) {
                const int k = gk + e;
                const bool valid = (unsigned)k < nlim;   // inside the window (k < 0 wraps) of an open event
                // == quantise(x, x0): scaling by 2^6 commutes with the rounding of the difference
                const int q = __float2int_rn(__fmaf_rn(row[g * kS + e], kQ, nx0));
                const int d = valid ? q - qa : 0;
                Sd += d; Sdd += (long long)d * d;
                const int cnt = valid ? k - k0 + 1 : 1;
                float rc = rct[min(cnt, kSeqTab - 1)];
                if (cnt >= kSeqTab) rc = __fdiv_rn(1.0f, (float)cnt);    // (a plateau beyond the table: rare)
                const float m = cusum_mean(Sd, rc);
                const float t = __fsub_rn((float)d, m);
                // quiet in every lane: the shortcut again (warp-uniform branch); the full evaluation is always valid
                const bool quiet = !valid || ((gp | gn) == 0 && fabsf(t) <= hq);
                if (__all_sync(CT_FULL, quiet)) { if (valid) { rp = k; rn = k; } continue; }
                const SeqOut s = cusum_tail(Sdd, m, rc, t, dq, hq);
                if (!valid) continue;
                // sums up to the last zero of each statistic (a statistic that is 0 now was last 0 at k - 1): what a
                // detection needs to cut the level at the changepoint without re-reading the samples behind it
                if (gp == 0) { ZpS = Sd - d; ZpSS = Sdd - (long long)d * d; }
                if (gn == 0) { ZnS = Sd - d; ZnSS = Sdd - (long long)d * d; }
                gp = max(gp + s.sp, 0); rp = gp == 0 ? k : rp;
                gn = max(gn + s.sn, 0); rn = gn == 0 ? k : rn;
                if (max(gp, gn) > H) {
                    if (nedge >= ML) {                       // level table full: the rest of the window is the last level
                        long long T = 0, TT = 0;
#pragma unroll 1
                        for (int j = e0; j < n; ++j) { const long long qj = quantise(a.y[p0 + j], x0); T += qj; TT += qj * qj; }
                        const long long r_ = (long long)ev * ML + (nedge - 1);
                        reinterpret_cast<long long*>(a.mean)[r_] = T;
                        reinterpret_cast<long long*>(a.sd)[r_] = TT;
                        a.edges[(long long)ev * (ML + 1) + nedge] = n;
                        a.n_levels[ev] = nedge;
                        a.overflow[ev] = (unsigned char)(1 | kRawSums);
                        running = false; nlim = 0u;
                        continue;
                    }
                    const bool pwin = gp >= gn;
                    const int edge = (pwin ? rp : rn) + 1;
                    const long long zs = pwin ? ZpS : ZnS, zss = pwin ? ZpSS : ZnSS;     // sums of d, d^2 over [k0, edge)
                    long long Aq, Aqq, Bq, Bqq;
                    level_sums(zs, zss, edge - k0, qa, Aq, Aqq);                                      // [k0, edge) in q units
                    level_sums(Sd - zs - d, Sdd - zss - (long long)d * d, k - edge, qa, Bq, Bqq);     // [edge, k)
                    const long long r_ = (long long)ev * ML + (nedge - 1);
                    CT_CHECK_RANGE(r_, 1, a.nev * ML, "cusum, level row");
                    reinterpret_cast<long long*>(a.mean)[r_] = Lp + Aq;           // level [e0, edge)
                    reinterpret_cast<long long*>(a.sd)[r_] = Lpp + Aqq;
                    a.edges[(long long)ev * (ML + 1) + nedge] = edge;
                    ++nedge;
                    e0 = edge; Lp = Bq; Lpp = Bqq;
                    k0 = k; qa = q; Sd = 0; Sdd = 0; gp = gn = 0; rp = rn = k;
                }
            }
            }
            if (act && running && gk + kS >= n) {            // the window ends in this group: level [e0, n)
                long long Sq, Sqq;
                level_sums(Sd, Sdd, n - k0, qa, Sq, Sqq);
                const long long r_ = (long long)ev * ML + (nedge - 1);
                reinterpret_cast<long long*>(a.mean)[r_] = Lp + Sq;
                reinterpret_cast<long long*>(a.sd)[r_] = Lpp + Sqq;
                a.edges[(long long)ev * (ML + 1) + nedge] = n;
                a.n_levels[ev] = nedge;
                a.overflow[ev] = kRawSums;
                running = false;
            }
        }
        __syncwarp();                                         // every lane is done with the rows of this stage
        fetch(stage);
        stage = stage + 1 == kStages ? 0 : stage + 1;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}

// ---- hand-out order: longest windows first -------------------------------------------------------------------
// Lanes take their next event from a shared counter, so the run ends when the lane that drew the last long window is
// done with it while its 31 neighbours idle.  Handing the windows out by decreasing length class (256 samples per
// class; a counting sort in two small kernels, the order inside a class is irrelevant: results are per event) leaves
// only the shortest windows for the end.
constexpr int kLenClasses = 64;
__device__ __forceinline__ int len_class(long long len) {
    if (len <= 0 || len > kSeqMax) return 0;                 // not for the lanes: dealt with at once
    const int c = (int)((len - 1) >> 8);
    return kLenClasses - 1 - (c < kLenClasses - 2 ? c : kLenClasses - 2);
}
__global__ void __launch_bounds__(256) ct_cusum_order_count(const long long* __restrict__ w0, const long long* __restrict__ w1,
                                                             long long nev, const long long* __restrict__ nev_dev,
                                                             unsigned* __restrict__ cls_count) {
    __shared__ unsigned h[kLenClasses];
    if (nev_dev) { const long long d = *nev_dev; nev = d < nev ? d : nev; }
    if (threadIdx.x < kLenClasses) h[threadIdx.x] = 0;
    __syncthreads();
    for (long long ev = (long long)blockIdx.x * blockDim.x + threadIdx.x; ev < nev; ev += (long long)gridDim.x * blockDim.x)
        atomicAdd(&h[len_class(w1[ev] - w0[ev])], 1u);
    __syncthreads();
    if (threadIdx.x < kLenClasses && h[threadIdx.x]) atomicAdd(&cls_count[threadIdx.x], h[threadIdx.x]);
}
__global__ void __launch_bounds__(256) ct_cusum_order_fill(const long long* __restrict__ w0, const long long* __restrict__ w1,
                                                            long long nev, const long long* __restrict__ nev_dev,
                                                            const unsigned* __restrict__ cls_count, unsigned* __restrict__ cls_fill,
                                                            int* __restrict__ order) {
    __shared__ unsigned base[kLenClasses], h[kLenClasses], off[kLenClasses];
    if (nev_dev) { const long long d = *nev_dev; nev = d < nev ? d : nev; }
    if (threadIdx.x == 0) {
        unsigned acc = 0;
        for (int c = 0; c < kLenClasses; ++c) { base[c] = acc; acc += cls_count[c]; }
    }
    constexpr int kChunk = 256 * 16;
    for (long long c0 = (long long)blockIdx.x * kChunk; c0 < nev; c0 += (long long)gridDim.x * kChunk) {
        __syncthreads();
        if (threadIdx.x < kLenClasses) h[threadIdx.x] = 0;
        __syncthreads();
        int cls[16]; unsigned pos[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const long long ev = c0 + i * 256 + threadIdx.x;
            cls[i] = -1;
            if (ev < nev) { cls[i] = len_class(w1[ev] - w0[ev]); pos[i] = atomicAdd(&h[cls[i]], 1u); }
        }
        __syncthreads();
        if (threadIdx.x < kLenClasses && h[threadIdx.x]) off[threadIdx.x] = base[threadIdx.x] + atomicAdd(&cls_fill[threadIdx.x], h[threadIdx.x]);
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 16; ++i)
            if (cls[i] >= 0) {
                CT_CHECK_RANGE(off[cls[i]] + pos[i], 1, nev, "cusum, hand-out order");
                order[off[cls[i]] + pos[i]] = (int)(c0 + i * 256 + threadIdx.x);
            }
    }
}

// float64 level mean / population std from the integer sums the lanes left in the arrays
// (oracle/events_oracle.py::level_stats, operation for operation).
__device__ __forceinline__ void finalize_level(const CusumArgs& a, long long i, double x0, int e0, int e1) {
    const double len = (double)(e1 - e0);
    const double ad = (double)reinterpret_cast<const long long*>(a.mean)[i];
    const double bd = (double)reinterpret_cast<const long long*>(a.sd)[i];
    a.mean[i] = __dadd_rn(x0, __ddiv_rn(__ddiv_rn(ad, len), 64.0));
    double var = __dsub_rn(bd, __ddiv_rn(__dmul_rn(ad, ad), len));
    if (var < 0.0) var = 0.0;
    a.sd[i] = __ddiv_rn(__dsqrt_rn(__ddiv_rn(var, len)), 64.0);
}
// One thread per event (any max_levels).
__global__ void ct_cusum_finalize_kernel(CusumArgs a) {
    long long nev = a.nev;
    if (a.nev_dev) { const long long d = *a.nev_dev; nev = d < nev ? d : nev; }
    const int ML = a.max_levels;
    for (long long ev = (long long)blockIdx.x * blockDim.x + threadIdx.x; ev < nev; ev += (long long)gridDim.x * blockDim.x) {
        const unsigned char f = a.overflow[ev];
        if (!(f & kRawSums)) continue;
        const int* ed = a.edges + ev * (ML + 1);
        const int nl = a.n_levels[ev];
        const double x0 = (double)a.y[a.w0[ev]];
        for (int lv = 0; lv < nl; ++lv) finalize_level(a, ev * ML + lv, x0, ed[lv], ed[lv + 1]);
        a.overflow[ev] = f & (unsigned char)~kRawSums;
    }
}
// One thread per table entry when max_levels divides the warp (the rows of the level table are then read and written
// as whole lines: 0.06 instead of 0.17 ms for 600 k events); an event's threads sit in one warp, so its flag is
// cleared once they have all read it.
__global__ void __launch_bounds__(256) ct_cusum_finalize_rows_kernel(CusumArgs a) {
    long long nev = a.nev;
    if (a.nev_dev) { const long long d = *a.nev_dev; nev = d < nev ? d : nev; }
    const int ML = a.max_levels;
    const long long total = nev * ML;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i0 = (long long)blockIdx.x * blockDim.x; i0 < total; i0 += stride) {
        const long long i = i0 + threadIdx.x;
        const bool in = i < total;
        const long long ev = in ? i / ML : 0;
        const int lv = (int)(i - ev * ML);
        unsigned char f = 0;
        int nl = 0;
        if (in) { f = a.overflow[ev]; nl = a.n_levels[ev]; }
        const bool raw = in && (f & kRawSums);
        if (raw && lv < nl) {
            const int* ed = a.edges + ev * (ML + 1);
            finalize_level(a, i, (double)a.y[a.w0[ev]], ed[lv], ed[lv + 1]);
        }
        __syncwarp();
        if (raw && lv == 0) a.overflow[ev] = f & (unsigned char)~kRawSums;
    }
}

// ---- per-event extrema of the window samples (max_deviation_pA of events.csv) ---------
__global__ void __launch_bounds__(256) ct_event_extrema_kernel(const float* __restrict__ y, long long ntot,
                                                                const long long* __restrict__ w0, const long long* __restrict__ w1,
                                                                long long nev, const long long* __restrict__ nev_dev,
                                                                float* __restrict__ xmin, float* __restrict__ xmax) {
    if (nev_dev) { const long long d = *nev_dev; nev = d < nev ? d : nev; }
    const int lane = ct_lane();
    const long long gw = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long ev = gw; ev < nev; ev += nw) {
        long long a = w0[ev], b = w1[ev];
        if (a < 0) a = 0;
        if (b > ntot) b = ntot;
        float lo = __int_as_float(0x7f800000), hi = __int_as_float(0xff800000);
        for (long long p = a + lane; p < b; p += 32) { const float v = y[p]; lo = fminf(lo, v); hi = fmaxf(hi, v); }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { lo = fminf(lo, __shfl_xor_sync(CT_FULL, lo, o)); hi = fmaxf(hi, __shfl_xor_sync(CT_FULL, hi, o)); }
        if (lane == 0) { xmin[ev] = lo; xmax[ev] = hi; }
    }
}

// ---- derived per-event statistics (the non-level columns of events.csv) ------------------------------
// mosaicConverter.py:72-154 derives them from the level list of an event; here one thread per event reads its rows
// of the level table (float64 means / stds from the exact integer sums, int32 edges) and leaves
//   cols[e][0..10] = baseline before, baseline after, effective baseline, sub-level duration (samples),
//                    average blockage, max blockage, its level's length (samples), min blockage, its level's
//                    length, residual (rms of trace minus step fit), max deviation from the effective baseline
// and the event's final type (0 accepted, 1 step-response fit, 5 CUSUM+ found no sub-level, 6 level overflow; other
// codes pass through).
// Conventions: cusumtools_b200/writer.py (blockage = sign(baseline) (baseline - level); in-event statistics run over
// the sub-levels 1 .. L-2; ties keep the first level).  Sums run level by level in index order.
constexpr int kEventCols = 12;
__global__ void ct_event_columns_kernel(const int* __restrict__ n_levels, const int* __restrict__ edges,
                                        const double* __restrict__ mean, const double* __restrict__ sd,
                                        const int* __restrict__ type, const unsigned char* __restrict__ overflow,
                                        const float* __restrict__ xmin, const float* __restrict__ xmax, long long nev,
                                        const long long* __restrict__ nev_dev, int ML, double* __restrict__ cols,
                                        int* __restrict__ type_out) {
    if (nev_dev) { const long long d = *nev_dev; nev = d < nev ? d : nev; }
    for (long long ev = (long long)blockIdx.x * blockDim.x + threadIdx.x; ev < nev; ev += (long long)gridDim.x * blockDim.x) {
        const int L = n_levels[ev];
        int t = type ? type[ev] : 0;
        // type 1 (step-response fit, level rows from ct_stepfit_batch) goes through the same arithmetic as type 0
        if ((t == 0 || t == 1) && overflow[ev]) t = 6;
        if ((t == 0 || t == 1) && L < 3) t = 5;
        type_out[ev] = t;
        double* c = cols + ev * kEventCols;
        if (t != 0 && t != 1) {
#pragma unroll
            for (int i = 0; i < kEventCols; ++i) c[i] = 0.0;
            continue;
        }
        const int* ed = edges + ev * (ML + 1);
        const double* mu = mean + ev * ML;
        const double* sg = sd + ev * ML;
        const double before = mu[0], after = mu[L - 1];
        const double eff = 0.5 * (before + after);
        const double sgn = eff >= 0.0 ? 1.0 : -1.0;
        double tot = 0.0, res = 0.0, dur = 0.0, wsum = 0.0;
        double bmax = -1.0 / 0.0, bmin = 1.0 / 0.0, lmax = 0.0, lmin = 0.0;
        for (int k = 0; k < L; ++k) {
            const double len = (double)(ed[k + 1] - ed[k]);
            tot += len;
            res += len * sg[k] * sg[k];
            if (k >= 1 && k < L - 1) {
                dur += len;
                wsum += len * mu[k];
                const double b = sgn * (eff - mu[k]);
                if (b > bmax) { bmax = b; lmax = len; }
                if (b < bmin) { bmin = b; lmin = len; }
            }
        }
        c[0] = before; c[1] = after; c[2] = eff; c[3] = dur;
        c[4] = sgn * (eff - wsum / dur);
        c[5] = bmax; c[6] = lmax; c[7] = bmin; c[8] = lmin;
        c[9] = sqrt(res / tot);
        c[10] = fmax(fabs((double)xmax[ev] - eff), fabs((double)xmin[ev] - eff));
        c[11] = 0.0;
    }
}

}  // namespace

extern "C" int ct_event_columns(const int32_t* n_levels, const int32_t* edges, const double* level_mean, const double* level_std,
                                const int32_t* type, const uint8_t* overflow, const float* xmin, const float* xmax,
                                int64_t n_events, const int64_t* n_events_dev, int max_levels, double* cols12, int32_t* type_out,
                                void* stream) {
    if (!n_levels || !edges || !level_mean || !level_std || !overflow || !xmin || !xmax || !cols12 || !type_out || n_events < 0 ||
        max_levels < 2) {
        ct_set_error("event_columns: bad argument"); return CT_ERR_ARG;
    }
    if (n_events == 0) return CT_OK;
    long long grid = (n_events + 255) / 256;
    const long long cap = (long long)ct_sm_count() * 8;
    if (grid > cap) grid = cap;
    CT_COUNT_LAUNCH();
    ct_event_columns_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(
        n_levels, edges, level_mean, level_std, type, overflow, xmin, xmax, n_events, (const long long*)n_events_dev, max_levels,
        cols12, type_out);
    return ct_check_launch("ct_event_columns_kernel");
}

// workspace: [0, 24) counters, [32, 544) class counts / fill counters of the hand-out order, then the pending list and
// the order (int32 per event each)
constexpr long long kWsHead = 32 + 2 * 4 * kLenClasses;
static long long ws_list_bytes(int64_t n_events) { return ((4 * (n_events > 0 ? n_events : 0)) + 15) & ~15LL; }
extern "C" int64_t ct_cusum_workspace_bytes(int64_t n_events) { return kWsHead + 2 * ws_list_bytes(n_events); }

static int cusum_launch(const float* y, int64_t n_total, const int64_t* win_start, const int64_t* win_end,
                        const int32_t* type, int64_t n_events, const int64_t* n_events_dev, float delta, float h,
                        int max_levels, int32_t* n_levels, int32_t* edges, double* level_mean, double* level_std,
                        uint8_t* overflow, void* workspace, int64_t workspace_bytes, void* stream) {
    if (!y || !win_start || !win_end || !n_levels || !edges || !level_mean || !level_std || !overflow || !workspace) {
        ct_set_error("cusum: null pointer"); return CT_ERR_ARG;
    }
    if (n_events < 0 || max_levels < 2 || max_levels > 1024 || !(delta > 0.f) || !(h > 0.f) || h > 262144.f) {
        ct_set_error("cusum: bad argument (need delta > 0, 0 < h <= 2^18, 2 <= max_levels <= 1024)"); return CT_ERR_ARG;
    }
    if (n_events > 0x7fffffffLL) { ct_set_error("cusum: more than 2^31-1 events in one batch"); return CT_ERR_UNSUPPORTED; }
    if (workspace_bytes < ct_cusum_workspace_bytes(n_events) || (reinterpret_cast<uintptr_t>(workspace) & 7)) {
        ct_set_error("cusum: workspace too small or unaligned"); return CT_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    cudaMemsetAsync(workspace, 0, kWsHead, st);
    if (n_events == 0) return CT_OK;
    CusumArgs a;
    a.y = y; a.ntot = n_total; a.w0 = (const long long*)win_start; a.w1 = (const long long*)win_end; a.type = type;
    a.nev = n_events; a.nev_dev = (const long long*)n_events_dev; a.delta = delta; a.h = h; a.max_levels = max_levels; a.n_levels = n_levels; a.edges = edges;
    a.mean = level_mean; a.sd = level_std; a.overflow = overflow; a.counter = (unsigned long long*)workspace;
    a.pending = reinterpret_cast<int*>((char*)workspace + kWsHead);
    a.order = nullptr;
    if (n_events >= kSeqMinEvents) {                         // (below that the warps take every event)
        unsigned* cls_count = reinterpret_cast<unsigned*>((char*)workspace + 32);
        unsigned* cls_fill = cls_count + kLenClasses;
        int* order = reinterpret_cast<int*>((char*)workspace + kWsHead + ws_list_bytes(n_events));
        long long og = (n_events + 256 * 16 - 1) / (256 * 16);
        if (og > 4LL * ct_sm_count()) og = 4LL * ct_sm_count();
        CT_COUNT_LAUNCH();
        ct_cusum_order_count<<<(unsigned)og, 256, 0, st>>>(a.w0, a.w1, n_events, a.nev_dev, cls_count);
        int rc0 = ct_check_launch("ct_cusum_order_count"); if (rc0) return rc0;
        CT_COUNT_LAUNCH();
        ct_cusum_order_fill<<<(unsigned)og, 256, 0, st>>>(a.w0, a.w1, n_events, a.nev_dev, cls_count, cls_fill, order);
        rc0 = ct_check_launch("ct_cusum_order_fill"); if (rc0) return rc0;
        a.order = order;
    }
    // rows of events nobody processes (rejected types) keep edges == -1
    cudaMemsetAsync(edges, 0xff, (size_t)n_events * (size_t)(max_levels + 1) * sizeof(int32_t), st);
    const int sms = ct_sm_count();
    int occ = 0;
    if (cudaFuncSetAttribute(ct_cusum_seq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSeqSmem) != cudaSuccess) {
        ct_set_error("cusum: cannot reserve %d bytes of shared memory", kSeqSmem); return CT_ERR_CUDA;
    }
    long long grid = sms;                                    // persistent: one CTA per SM
    long long want = (n_events + kSeqWarps * 32 - 1) / (kSeqWarps * 32);
    if (grid > want) grid = want;
    CT_COUNT_LAUNCH();
    ct_cusum_seq_kernel<<<(unsigned)grid, kSeqWarps * 32, kSeqSmem, st>>>(a);
    int rc = ct_check_launch("ct_cusum_seq_kernel"); if (rc) return rc;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ct_cusum_warp_kernel, 128, 0);
    if (occ < 1) occ = 1;
    grid = (long long)sms * occ;
    want = (n_events + 3) / 4;
    if (grid > want) grid = want;
    CT_COUNT_LAUNCH();
    ct_cusum_warp_kernel<<<(unsigned)grid, 128, 0, st>>>(a);
    rc = ct_check_launch("ct_cusum_warp_kernel"); if (rc) return rc;
    CT_COUNT_LAUNCH();
    if (max_levels <= 32 && 32 % max_levels == 0) {
        grid = (n_events * max_levels + 255) / 256;
        if (grid > (long long)sms * 8) grid = (long long)sms * 8;
        ct_cusum_finalize_rows_kernel<<<(unsigned)grid, 256, 0, st>>>(a);
    } else {
        grid = (n_events + 255) / 256;
        if (grid > (long long)sms * 8) grid = (long long)sms * 8;
        ct_cusum_finalize_kernel<<<(unsigned)grid, 256, 0, st>>>(a);
    }
    return ct_check_launch("ct_cusum_finalize_kernel");
}

extern "C" int ct_cusum_batch(const float* y, int64_t n_total, const int64_t* win_start, const int64_t* win_end,
                              const int32_t* type, int64_t n_events, float delta, float h, int max_levels,
                              int32_t* n_levels, int32_t* edges, double* level_mean, double* level_std,
                              uint8_t* overflow, void* workspace, int64_t workspace_bytes, void* stream) {
    return cusum_launch(y, n_total, win_start, win_end, type, n_events, nullptr, delta, h, max_levels, n_levels, edges,
                        level_mean, level_std, overflow, workspace, workspace_bytes, stream);
}

extern "C" int ct_cusum_batch_dev(const float* y, int64_t n_total, const int64_t* win_start, const int64_t* win_end,
                                  const int32_t* type, const int64_t* n_events_dev, int64_t capacity, float delta,
                                  float h, int max_levels, int32_t* n_levels, int32_t* edges, double* level_mean,
                                  double* level_std, uint8_t* overflow, void* workspace, int64_t workspace_bytes,
                                  void* stream) {
    if (!n_events_dev) { ct_set_error("cusum: null event count pointer"); return CT_ERR_ARG; }
    return cusum_launch(y, n_total, win_start, win_end, type, capacity, n_events_dev, delta, h, max_levels, n_levels,
                        edges, level_mean, level_std, overflow, workspace, workspace_bytes, stream);
}

extern "C" int ct_event_extrema_f32(const float* y, int64_t n_total, const int64_t* win_start, const int64_t* win_end,
                                    int64_t n_events, const int64_t* n_events_dev, float* xmin, float* xmax, void* stream) {
    if (!y || !win_start || !win_end || !xmin || !xmax || n_events < 0) { ct_set_error("event_extrema: bad argument"); return CT_ERR_ARG; }
    if (n_events == 0) return CT_OK;
    long long grid = (n_events + 7) / 8;
    const long long cap = (long long)ct_sm_count() * 8;
    if (grid > cap) grid = cap;
    CT_COUNT_LAUNCH();
    ct_event_extrema_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(
        y, n_total, (const long long*)win_start, (const long long*)win_end, n_events, (const long long*)n_events_dev, xmin, xmax);
    return ct_check_launch("ct_event_extrema_kernel");
}
